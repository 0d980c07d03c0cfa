// primitives.cuh — device-wide building blocks used by the graph build and
// CORE-A stages: a generic single-pass prefix scan (also used as stream
// compaction) and an LSD radix sort of 64-bit keys (sort.cu).  All HBM-bound integer work.
#pragma once

#include "common.cuh"

namespace kg {

// One radix pass sorts on a digit of at most 8 bits: key bits [shift, shift+bits), and above them (when bits2 > 0)
// key bits [shift2, shift2+bits2) -- a digit may straddle the gap between two key fields, so that e.g. a
// (20 + 20)-bit pair key takes 5 passes of 8 bits instead of 3 + 3 passes of 7.
struct RadixPass {
    int shift;
    int bits;
    int shift2;
    int bits2;
};

// Split the key bit ranges [lo0,hi0) and [lo1,hi1) (second may be empty), read as one bit string, into the
// fewest passes of at most 8 bits (equal widths), least significant first.
int plan_radix_passes(int lo0, int hi0, int lo1, int hi1, RadixPass *out /* >= 8 entries */);

// What a sort may take besides its keys, all optional.
struct SortOptions {
    // Pass 1 reads the keys here and leaves them unchanged; `a` is then only scratch (needed from 3 passes on, or
    // from 2 without `col`).
    const uint64_t *first = nullptr;
    // counts[x], x < n_counts: the number of keys whose low word is x, when every pass's digit lies in the low word.
    // The digit histograms come from these instead of from a read of the keys.
    const uint32_t *counts = nullptr;
    uint32_t n_counts = 0;
    // The last pass writes no keys: the key (hi << 32 | lo) at sorted position pos stores hi at col[col_base[lo] + pos]
    // (the back half of every CSR row, keys sorted on lo).  With fewer than 2 keys or no passes they go there unsorted.
    const uint32_t *col_base = nullptr;
    uint32_t *col = nullptr;
    // With col: pass 1 (or, without passes, the unsorted store) also writes the forward half of every row as it reads
    // the keys, which are then the u-sorted edge list with col_base its row starts: key i = (u << 32 | v) stores v at
    // col[i + fwd_row_ptr[u + 1] - col_base[u + 1]].
    const uint64_t *fwd_row_ptr = nullptr;
};

// Stable LSD radix sort.  `a` holds the keys, `b` is scratch of the same size;
// returns in *sorted whichever of the two holds the result (nullptr when opt->col takes it).
int radix_sort_u64(kombgpu_ctx *ctx, uint64_t *a, uint64_t *b, uint64_t n, const RadixPass *passes,
                   int n_passes, uint64_t **sorted, const SortOptions *opt = nullptr);

#ifdef __CUDACC__

constexpr int kScanThreads = 512;

// Single-pass scan (chained scan with decoupled look-back): every element's in(i) is evaluated ONCE (some of the
// path's functors look back through a read or compare neighbouring keys) and every access stays coalesced (item j of
// thread t is element base + j * threads + t).  Inside a tile: one warp scan per item, the 16 x 16 (item, warp)
// totals scanned once by the CTA -- two barriers a tile, not three per item.  Tiles
// take their index from a counter and learn the sum of all earlier tiles from 64-bit status words (2 flag bits +
// 62-bit value: every sum on this path is far below 2^62), 32 predecessors per look-back step.
constexpr uint64_t kScanFlagAgg = 1ull << 62, kScanFlagPrefix = 2ull << 62, kScanValueMask = (1ull << 62) - 1;
template <typename T> struct ScanShape { static constexpr int kItems = sizeof(T) > 4 ? 8 : 16; };   // registers: v[] + wex[]

template <typename T, typename InFn, typename OutFn>
__global__ void __launch_bounds__(kScanThreads) scan_onepass_kernel(uint64_t n, InFn in, OutFn out, uint64_t *status,
                                                                    uint32_t *tile_counter, uint32_t n_tiles, T *total) {
    constexpr int kItems = ScanShape<T>::kItems;
    constexpr int kWarps = kScanThreads / 32;
    __shared__ T s_tot[kItems * kWarps];
    __shared__ T s_scan[kWarps + 1];
    __shared__ uint64_t s_excl;
    __shared__ uint32_t s_tile;
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_tile = atomicAdd(tile_counter, 1u);
    __syncthreads();
    const uint32_t tile = s_tile;
    const uint64_t base = (uint64_t)tile * (kScanThreads * kItems);
    T v[kItems], wex[kItems];
#pragma unroll
    for (int j = 0; j < kItems; ++j) {
        const uint64_t i = base + (uint64_t)j * kScanThreads + threadIdx.x;
        v[j] = i < n ? in(i) : T(0);
    }
#pragma unroll
    for (int j = 0; j < kItems; ++j) {
        const T incl = warp_incl_scan_add(v[j]);
        wex[j] = incl - v[j];
        if (lane == 31) s_tot[j * kWarps + warp] = incl;
    }
    __syncthreads();
    // (item, warp) totals in element order: item-major
    const T mine = threadIdx.x < kItems * kWarps ? s_tot[threadIdx.x] : T(0);
    T tile_total;
    const T off = block_excl_scan_add<T, kScanThreads>(mine, s_scan, &tile_total);
    if (threadIdx.x < kItems * kWarps) s_tot[threadIdx.x] = off;
    if (threadIdx.x < 32) {
        uint64_t excl = 0;
        if (lane == 0)
            asm volatile("st.volatile.global.u64 [%0], %1;" ::"l"(status + tile),
                         "l"((tile == 0 ? kScanFlagPrefix : kScanFlagAgg) | (uint64_t)tile_total) : "memory");
        if (tile > 0) {
            int64_t p = (int64_t)tile - 1;   // lane l looks at tile p - l
            while (true) {
                const int64_t idx = p - (int64_t)lane;
                uint64_t w = kScanFlagPrefix;   // before tile 0: an empty prefix
                if (idx >= 0) {
                    uint32_t spins = 0;
                    do {
                        asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(w) : "l"(status + idx) : "memory");
                        if (++spins > (1u << 28)) __trap();
                    } while ((w >> 62) == 0);
                }
                const uint32_t pm = __ballot_sync(kFullMask, (w & kScanFlagPrefix) != 0);
                // tiles p .. p - f contribute (f = nearest predecessor that already knows its inclusive prefix)
                const uint32_t f = pm ? (uint32_t)__ffs(pm) - 1u : 31u;
                uint64_t part = lane <= f ? (w & kScanValueMask) : 0ull;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(kFullMask, part, o);
                excl += part;
                if (pm) break;
                p -= 32;
            }
            if (lane == 0)
                asm volatile("st.volatile.global.u64 [%0], %1;" ::"l"(status + tile), "l"(kScanFlagPrefix | (excl + (uint64_t)tile_total))
                             : "memory");
        }
        if (lane == 0) {
            s_excl = excl;
            if (tile == n_tiles - 1 && total) *total = (T)(excl + (uint64_t)tile_total);
        }
    }
    __syncthreads();
    const T tile_base = (T)s_excl;
#pragma unroll
    for (int j = 0; j < kItems; ++j) {
        const uint64_t i = base + (uint64_t)j * kScanThreads + threadIdx.x;
        if (i < n) out(i, tile_base + s_tot[j * kWarps + warp] + wex[j], v[j]);
    }
}

// Exclusive prefix sum over in(0..n-1); out(i, prefix, value) is called once per
// element; *total_dev (device, optional) receives the grand total.
template <typename T, typename InFn, typename OutFn>
int device_scan(kombgpu_ctx *ctx, uint64_t n, InFn in, OutFn out, T *total_dev) {
    if (n == 0) {
        if (total_dev) KG_CUDA(ctx, cudaMemsetAsync(total_dev, 0, sizeof(T), ctx->stream));
        return KOMBGPU_OK;
    }
    const uint32_t n_tiles = ceil_div_u64(n, (uint64_t)kScanThreads * ScanShape<T>::kItems);
    DevBuf<uint64_t> status;   // [n_tiles status words | tile counter]
    KG_ALLOC(ctx, status, (size_t)n_tiles + 1);
    KG_CUDA(ctx, cudaMemsetAsync(status.p, 0, ((size_t)n_tiles + 1) * sizeof(uint64_t), ctx->stream));
    KG_LAUNCH(ctx, (scan_onepass_kernel<T, InFn, OutFn>), n_tiles, kScanThreads, 0, n, in, out, status.p,
              reinterpret_cast<uint32_t *>(status.p + n_tiles), n_tiles, total_dev);
    return KOMBGPU_OK;
}

// functors shared by several stages ------------------------------------------------

// head-of-run predicate on a sorted key array: 1 when keys[i] != keys[i-1]
struct HeadFlagU64 {
    const uint64_t *keys;
    __device__ uint32_t operator()(uint64_t i) const { return (i == 0 || keys[i] != keys[i - 1]) ? 1u : 0u; }
};
// write keys[i] to dst[prefix] when flagged: adjacent-unique of a sorted array
struct CompactKeysU64 {
    const uint64_t *keys;
    uint64_t *dst;
    __device__ void operator()(uint64_t i, uint32_t pos, uint32_t flag) const {
        if (flag) dst[pos] = keys[i];
    }
};

#endif  // __CUDACC__

}  // namespace kg
