// extend.cu — the list merge of Extend (pyrope_index_extend): append the write buffer's rows to the inverted lists of a
// built IVF index without re-training.  The host side (api.cu) assigns the buffered rows to the current centroids,
// encodes them with the current codebooks and groups them by list (group_by_cluster, a stable sort); this kernel then
// writes every merged list array in one pass:
//   merged list c starts at off_old[c] + offs_new[c];
//   old entry i of list c (list-major position i) lands at i + offs_new[c]   (a contiguous run per list, shifted);
//   new sorted entry j of list c lands at off_old[c + 1] + j                  (gathered from buffer order via `order`).
// The grid walks the DESTINATION arrays in fixed 16 KiB tiles, so a skewed list is split over as many CTAs as its bytes
// need and many short lists share one CTA; each CTA finds its first list by binary search over the merged offsets.
#include <cstdint>

#include "kernels.h"

namespace pyrope {
namespace {

constexpr int kThreads = 256;
constexpr int64_t kTileBytes = 16384;  // bytes of one column one CTA writes (a multiple of 16)

// 16 bytes starting r bytes into the 32-byte little-endian concatenation a:b
__device__ __forceinline__ uint4 shift_pair(const uint4 a, const uint4 b, int r) {
    const int q = r >> 2;
    const unsigned sh = (unsigned)(r & 3) * 8u;
    const uint32_t y0 = q == 0 ? a.x : q == 1 ? a.y : q == 2 ? a.z : a.w;
    const uint32_t y1 = q == 0 ? a.y : q == 1 ? a.z : q == 2 ? a.w : b.x;
    const uint32_t y2 = q == 0 ? a.z : q == 1 ? a.w : q == 2 ? b.x : b.y;
    const uint32_t y3 = q == 0 ? a.w : q == 1 ? b.x : q == 2 ? b.y : b.z;
    const uint32_t y4 = q == 0 ? b.x : q == 1 ? b.y : q == 2 ? b.z : b.w;
    return make_uint4(__funnelshift_r(y0, y1, sh), __funnelshift_r(y1, y2, sh), __funnelshift_r(y2, y3, sh),
                      __funnelshift_r(y3, y4, sh));
}

// dead flags hold 0..3 (1 deleted, 2 shadowed): every non-zero byte becomes 1
__device__ __forceinline__ uint32_t fold_word(uint32_t w) { return (w | (w >> 1)) & 0x01010101u; }
__device__ __forceinline__ uint4 fold4(uint4 v) { return make_uint4(fold_word(v.x), fold_word(v.y), fold_word(v.z), fold_word(v.w)); }

// dst bytes [a, z) of a column take src bytes [a - shift, z - shift).  dst is 16-byte aligned (cudaMalloc); src may sit
// at any byte offset against it (IVF_PQ rows are m bytes): aligned 16-byte stores, each fed by the one or two aligned
// 16-byte source words it overlaps.  The unaligned head and tail of the run go byte by byte.
__device__ __forceinline__ void copy_run(uint8_t* __restrict__ dst, const uint8_t* __restrict__ src, int64_t a, int64_t z,
                                         int64_t shift, bool fold) {
    const int64_t wa = (a + 15) & ~(int64_t)15, wz = z & ~(int64_t)15;
    if (wa >= wz) {
        for (int64_t x = a + threadIdx.x; x < z; x += kThreads) {
            const uint8_t v = src[x - shift];
            dst[x] = fold ? (uint8_t)(v != 0) : v;
        }
        return;
    }
    const int64_t nh = wa - a, nt = z - wz;
    for (int64_t t = threadIdx.x; t < nh + nt; t += kThreads) {
        const int64_t x = t < nh ? a + t : wz + (t - nh);
        const uint8_t v = src[x - shift];
        dst[x] = fold ? (uint8_t)(v != 0) : v;
    }
    const uintptr_t sbase = (uintptr_t)src - (uintptr_t)shift;
    for (int64_t w = wa + (int64_t)threadIdx.x * 16; w < wz; w += (int64_t)kThreads * 16) {
        const uintptr_t s = sbase + (uintptr_t)w;
        const int r = (int)(s & 15);
        const uint4* p = reinterpret_cast<const uint4*>(s - (uintptr_t)r);
        const uint4 lo = __ldg(p);
        uint4 v = lo;
        if (r) v = shift_pair(lo, __ldg(p + 1), r);  // both words hold bytes of the run: the dst word lies inside it
        if (fold) v = fold4(v);
        *reinterpret_cast<uint4*>(dst + w) = v;
    }
}

// dst bytes [a, z) of the new part of list c, which starts at byte mo: entry e = (x - mo) / rb of that part is buffer
// row order[sorted0 + e].  W-byte words (W divides rb, and a, z, mo are multiples of W).  src == nullptr writes zeros.
template <typename T>
__device__ __forceinline__ void copy_new(uint8_t* __restrict__ dst, const uint8_t* __restrict__ src, int64_t a, int64_t z,
                                         int64_t mo, int64_t rb, int64_t sorted0, const int32_t* __restrict__ order) {
    constexpr int W = (int)sizeof(T);
    for (int64_t x = a + (int64_t)threadIdx.x * W; x < z; x += (int64_t)kThreads * W) {
        T v;
        if (src) {
            const int64_t rel = x - mo, e = rel / rb, o = rel - e * rb;
            const int64_t row = order[sorted0 + e];
            v = *reinterpret_cast<const T*>(src + row * rb + o);
        } else {
            v = T{};
        }
        *reinterpret_cast<T*>(dst + x) = v;
    }
}

__global__ void __launch_bounds__(kThreads) extend_merge_lists_kernel(const ExtendMergeParams p) {
    const int64_t b = blockIdx.x;
    ExtendMergeColumn c = p.col[0];
#pragma unroll
    for (int i = 1; i < kExtendMaxColumns; ++i)
        if (i < p.ncols && b >= p.col[i].tile0) c = p.col[i];
    const int64_t rb = c.row_bytes;
    const int nc = p.nc;
    const int64_t t0 = (b - c.tile0) * kTileBytes;
    const int64_t t1 = min(t0 + kTileBytes, p.off_merged[nc] * rb);
    __shared__ int s_first;
    if (threadIdx.x == 0) {  // first list whose merged range ends after the tile's first entry
        const int64_t e0 = t0 / rb;
        int lo = 0, hi = nc - 1;
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (p.off_merged[mid + 1] > e0) hi = mid;
            else lo = mid + 1;
        }
        s_first = lo;
    }
    __syncthreads();
    for (int l = s_first; l < nc; ++l) {
        const int64_t m0 = p.off_merged[l] * rb;
        if (m0 >= t1) break;
        const int64_t m1 = p.off_merged[l + 1] * rb;
        const int64_t o0 = p.off_old[l];
        const int64_t mo = m0 + (p.off_old[l + 1] - o0) * rb;  // end of the old run in the merged array
        int64_t a = max(t0, m0), z = min(t1, mo);
        if (a < z) copy_run(c.dst, c.old_src, a, z, m0 - o0 * rb, c.fold_flags != 0);
        a = max(t0, mo);
        z = min(t1, m1);
        if (a < z) {
            const int64_t s0 = p.offs_new[l];
            if (rb % 16 == 0) copy_new<uint4>(c.dst, c.new_src, a, z, mo, rb, s0, p.order);
            else if (rb % 4 == 0) copy_new<uint32_t>(c.dst, c.new_src, a, z, mo, rb, s0, p.order);
            else copy_new<uint8_t>(c.dst, c.new_src, a, z, mo, rb, s0, p.order);
        }
    }
}

}  // namespace

int64_t extend_merge_tiles(int64_t merged_rows, int64_t row_bytes) { return (merged_rows * row_bytes + kTileBytes - 1) / kTileBytes; }

cudaError_t launch_extend_merge(ExtendMergeParams p, int64_t merged_rows, cudaStream_t st) {
    if (p.ncols < 1 || p.ncols > kExtendMaxColumns || p.nc < 1) return cudaErrorInvalidValue;
    int64_t tiles = 0;
    for (int i = 0; i < p.ncols; ++i) {
        p.col[i].tile0 = tiles;
        tiles += extend_merge_tiles(merged_rows, p.col[i].row_bytes);
    }
    for (int i = p.ncols; i < kExtendMaxColumns; ++i) p.col[i].tile0 = INT64_MAX;
    if (tiles == 0) return cudaSuccess;
    if (tiles >= ((int64_t)1 << 31)) return cudaErrorInvalidValue;
    extend_merge_lists_kernel<<<(unsigned)tiles, kThreads, 0, st>>>(p);
    return cudaGetLastError();
}

}  // namespace pyrope
