// sort.cu — stable LSD radix sort of 64-bit keys (unitig pairs, edges by their second endpoint, CORE-A rank keys, and
// hits when they do not arrive in read order).  Integer, HBM-bound.
//
// Single-read passes (radix_sweep_kernel, "onesweep"): one kernel histograms every pass's digit up front, then each
// pass reads the keys once and writes them once; tiles learn their global offsets by a decoupled look-back over
// per-tile status words.  The tile is staged in shared memory in digit order so global stores are contiguous runs.
// One implementation serves every n < 2^32: only the width of the status words depends on n (see StatusWord).
// What bounds a pass is instruction issue, not DRAM: ~130 thread-instructions per key, half of them the
// ballot-per-digit-bit ranking (profiles/r1/r1o_sweep_*).  MATCH.ANY ranks a key in one instruction but runs on the ADU
// pipe and made every mix of the two slower (round 1).  Measurements of the passes and of the tile geometries that lost
// to the one below are in DESIGN.md §4 "Sort".
#include <type_traits>

#include "kombgpu_debug.h"
#include "primitives.cuh"

namespace kg {

namespace {

constexpr int kRsThreads = 512;
constexpr int kRsItems = 8;
constexpr int kRsTile = kRsThreads * kRsItems;  // 4096 keys per CTA of the histogram kernel
constexpr int kRadix = 256;
constexpr int kMaxPasses = 8;

// digit extraction of one pass (RadixPass)
struct DigitSpec {
    int shift, shift2, bits1;
    uint32_t mask1, mask2, mask;   // mask = all digit bits
    __host__ __device__ static DigitSpec of(const RadixPass &p) {
        DigitSpec d;
        d.shift = p.shift; d.shift2 = p.shift2; d.bits1 = p.bits;
        d.mask1 = (1u << p.bits) - 1u; d.mask2 = (1u << p.bits2) - 1u;
        d.mask = (1u << (p.bits + p.bits2)) - 1u;
        return d;
    }
    __device__ __forceinline__ uint32_t operator()(uint64_t key) const {
        return ((uint32_t)(key >> shift) & mask1) | (((uint32_t)(key >> shift2) & mask2) << bits1);
    }
};

// ---------------------------------------------------------------------------
// Single-read passes ("onesweep": Adinets & Merrill 2022).  One kernel up front
// histograms every pass's digit (one read of the keys); each pass is then ONE
// kernel that reads the keys once and writes them once.  A tile (CTA) takes its
// index from a counter (so every predecessor is already running), ranks its keys,
// publishes its 256 digit counts as (AGGREGATE | count) words, and finds the number
// of keys with the same digit in earlier tiles by walking back over its
// predecessors' words until it meets one marked (PREFIX | inclusive count)
// (decoupled look-back); then it publishes its own PREFIX words.  In steady state a
// walk ends after one or two hops, because predecessors started earlier.
// ---------------------------------------------------------------------------

// Look-back status word: 2 flag bits above a count.  uint32_t holds counts below 2^30, so it serves n < 2^30 keys;
// longer arrays, where one digit's inclusive count can pass 2^30, take uint64_t (62-bit counts, the split of
// scan_onepass_kernel's words).  Counts themselves stay below n < 2^32.
template <typename W>
struct StatusWord {
    static constexpr int kShift = 8 * (int)sizeof(W) - 2;
    static constexpr W kAgg = W(1) << kShift, kPrefix = W(2) << kShift, kValueMask = (W(1) << kShift) - 1;
    // volatile accesses (other CTAs write these words during the launch), as width-specific inline asm
    static __device__ __forceinline__ W load(const W *p) {
        W w;
        if constexpr (sizeof(W) == 4) asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(w) : "l"(p) : "memory");
        else asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(w) : "l"(p) : "memory");
        return w;
    }
    static __device__ __forceinline__ void store(W *p, W w) {
        if constexpr (sizeof(W) == 4) asm volatile("st.volatile.global.u32 [%0], %1;" ::"l"(p), "r"(w) : "memory");
        else asm volatile("st.volatile.global.u64 [%0], %1;" ::"l"(p), "l"(w) : "memory");
    }
};

struct PassList {
    DigitSpec dg[kMaxPasses];
    int n;
};

// hist[p * 256 + d] += number of keys whose pass-p digit is d
__global__ void __launch_bounds__(kRsThreads) radix_global_hist_kernel(const uint64_t *__restrict__ keys, uint64_t n, PassList pl,
                                                                       uint32_t *__restrict__ hist) {
    __shared__ uint32_t s_hist[kMaxPasses * kRadix];
    for (int i = threadIdx.x; i < pl.n * kRadix; i += kRsThreads) s_hist[i] = 0;
    __syncthreads();
    const uint32_t lane = lane_id();
    for (uint64_t base = (uint64_t)blockIdx.x * kRsTile; base < n; base += (uint64_t)gridDim.x * kRsTile) {
        uint64_t key[kRsItems];
#pragma unroll
        for (int j = 0; j < kRsItems; ++j) {
            const uint64_t i = base + (uint64_t)j * kRsThreads + threadIdx.x;
            key[j] = i < n ? keys[i] : ~0ull;
        }
#pragma unroll
        for (int j = 0; j < kRsItems; ++j) {
            const uint64_t i = base + (uint64_t)j * kRsThreads + threadIdx.x;
            const bool valid = i < n;
            const bool full = __all_sync(kFullMask, valid);
            for (int p = 0; p < pl.n; ++p) {
                const uint32_t d = pl.dg[p](key[j]);
                // sorted or narrow digits put a whole warp on one counter: count it once
                const uint32_t d0 = __shfl_sync(kFullMask, d, 0);
                if (full && __all_sync(kFullMask, d == d0)) {
                    if (lane == 0) atomicAdd(&s_hist[p * kRadix + d0], 32u);
                } else if (valid) {
                    atomicAdd(&s_hist[p * kRadix + d], 1u);
                }
            }
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < pl.n * kRadix; i += kRsThreads)
        if (s_hist[i]) atomicAdd(&hist[i], s_hist[i]);
}

// exclusive prefix over the 256 digits of every pass (one CTA per pass, 256 threads)
__global__ void __launch_bounds__(kRadix) radix_hist_scan_kernel(uint32_t *hist) {
    __shared__ uint32_t s_tmp[kRadix / 32 + 1];
    uint32_t *h = hist + (size_t)blockIdx.x * kRadix;
    const uint32_t v = h[threadIdx.x];
    uint32_t total = 0;
    const uint32_t ex = block_excl_scan_add<uint32_t, kRadix>(v, s_tmp, &total);
    h[threadIdx.x] = ex;
}

// Tile of the sweep kernel: 512 threads x 16 keys, 2 CTAs per SM.  The per-digit phases (prefix over warps, look-back)
// are amortised over more keys than in the smaller tiles measured against it (DESIGN.md §4 "Sort").
constexpr int kSweepThreads = 512, kSweepItems = 16, kSweepTile = kSweepThreads * kSweepItems, kSweepMinBlocks = 2;

struct SweepSmem {
    uint64_t keys[kSweepTile];
    uint32_t warp_cnt[kSweepThreads / 32][kRadix];
    uint32_t digit_local[kRadix];   // first slot of digit d inside the staged tile
    uint32_t digit_global[kRadix];  // global position of that slot minus digit_local
    uint32_t digit_total[kRadix];
    uint32_t tile;
};

// Where a pass puts key k at its sorted position pos: every pass but a sink's last one writes the key array `out`.
struct StoreKeys {
    __device__ __forceinline__ void operator()(uint64_t *__restrict__ out, uint64_t pos, uint64_t k) const { out[pos] = k; }
};
// The CSR's back half (SortOptions::col): the v-sorted edge (u << 32 | v) at position pos is u, at col[col_base[v] + pos]
struct StoreCol {
    const uint32_t *col_base;
    uint32_t *col;
    __device__ __forceinline__ void operator()(uint64_t *, uint64_t pos, uint64_t k) const {
        col[(uint64_t)col_base[(uint32_t)k] + pos] = (uint32_t)(k >> 32);
    }
};

// What the first pass may do with each key it reads, besides sorting it (SortOptions::fwd_row_ptr)
struct NoVisit {};
// The CSR's forward half: edge i = (u << 32 | v) of the u-sorted list is v, at col[i + row_ptr[u + 1] - col_base[u + 1]]
struct VisitFwdCol {
    const uint64_t *row_ptr;
    const uint32_t *col_base;
    uint32_t *col;
    __device__ __forceinline__ void operator()(uint64_t i, uint64_t k) const {
        const uint32_t u1 = (uint32_t)(k >> 32) + 1u;
        col[i + row_ptr[u1] - col_base[u1]] = (uint32_t)k;
    }
};

// W: status word (StatusWord).  kBits: digit width known at compile time (8), or 0 = read it from `mask`.
// Store: where the sorted keys go (StoreKeys, or StoreCol in the last pass of a CSR sort).  Visit: called on every key
// as it is read (NoVisit, or VisitFwdCol in the first pass of a CSR sort).
template <typename W, int kBits, typename Store, typename Visit>
__global__ void __launch_bounds__(kSweepThreads, kSweepMinBlocks) radix_sweep_kernel(const uint64_t *__restrict__ in, uint64_t *__restrict__ out,
                                                                    uint64_t n, DigitSpec dg,
                                                                    const uint32_t *__restrict__ digit_base,  // exclusive global histogram of this pass
                                                                    W *status, uint32_t *tile_counter, Store store, Visit visit) {
    using SW = StatusWord<W>;
    constexpr int kWarps = kSweepThreads / 32;
    extern __shared__ __align__(16) unsigned char s_raw[];
    SweepSmem &s = *reinterpret_cast<SweepSmem *>(s_raw);
    const uint32_t warp = threadIdx.x >> 5, lane = lane_id();
    const uint32_t mask = kBits ? (1u << kBits) - 1u : dg.mask;
    if (threadIdx.x == 0) s.tile = atomicAdd(tile_counter, 1u);
    for (int i = threadIdx.x; i < kWarps * kRadix; i += kSweepThreads) (&s.warp_cnt[0][0])[i] = 0;
    __syncthreads();
    const uint32_t tile = s.tile;
    const uint64_t tile_base = (uint64_t)tile * kSweepTile;
    const uint32_t tile_count = (uint32_t)min((uint64_t)kSweepTile, n - tile_base);

    // warp-striped load: item j of lane l is tile element warp*32*kSweepItems + j*32 + l, so (warp, j, lane) order is
    // memory order and the sort stays stable
    uint64_t key[kSweepItems];
    uint16_t rank[kSweepItems];
    const uint32_t warp_base = warp * (32 * kSweepItems);
#pragma unroll
    for (int j = 0; j < kSweepItems; ++j) {
        const uint32_t e = warp_base + j * 32 + lane;
        key[j] = e < tile_count ? in[tile_base + e] : 0;
    }
    // rank inside the warp: lanes with the same digit are found with one ballot per digit bit; the group's leader takes
    // the digit's running count with a shared-memory atomic (issued in j order: stable)
#pragma unroll
    for (int j = 0; j < kSweepItems; ++j) {
        const uint32_t e = warp_base + j * 32 + lane;
        const bool valid = e < tile_count;
        const uint32_t d = valid ? dg(key[j]) : 0u;
        uint32_t same = __ballot_sync(kFullMask, valid);
#pragma unroll
        for (int b = 0; b < 8; ++b) {
            if (kBits ? (b >= kBits) : ((mask >> b) == 0)) break;  // uniform: narrower digits need fewer ballots
            const uint32_t bit = (d >> b) & 1u;
            const uint32_t vote = __ballot_sync(kFullMask, bit);
            same &= vote ^ (bit - 1u);   // lanes whose bit equals mine
        }
        const uint32_t lead = valid ? (uint32_t)__ffs(same) - 1u : lane;
        uint32_t base = 0;
        if (valid && lead == lane) base = atomicAdd(&s.warp_cnt[warp][d], (uint32_t)__popc(same));
        rank[j] = (uint16_t)(__popc(same & lanemask_lt()) + __shfl_sync(kFullMask, base, lead));
    }
    __syncthreads();

    // per digit: exclusive prefix over warps; publish the tile's count (the look-back starts from it)
    for (uint32_t d = threadIdx.x; d < (uint32_t)kRadix; d += kSweepThreads) {
        uint32_t total = 0;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) {
            const uint32_t c = s.warp_cnt[w][d];
            s.warp_cnt[w][d] = total;
            total += c;
        }
        s.digit_total[d] = total;
        if (d <= mask) SW::store(status + (size_t)tile * kRadix + d, (tile == 0 ? SW::kPrefix : SW::kAgg) | (W)total);
    }
    __syncthreads();
    if (warp == 0) {   // exclusive scan of the 256 digit totals: 8 per lane
        uint32_t v[kRadix / 32], sum = 0;
#pragma unroll
        for (int i = 0; i < kRadix / 32; ++i) { v[i] = s.digit_total[lane * (kRadix / 32) + i]; sum += v[i]; }
        uint32_t run = warp_incl_scan_add(sum) - sum;
#pragma unroll
        for (int i = 0; i < kRadix / 32; ++i) { s.digit_local[lane * (kRadix / 32) + i] = run; run += v[i]; }
    }
    __syncthreads();

    // stage the tile in digit order (the look-back follows, overlapping other CTAs' work)
#pragma unroll
    for (int j = 0; j < kSweepItems; ++j) {
        const uint32_t e = warp_base + j * 32 + lane;
        if (e < tile_count) {
            const uint32_t d = dg(key[j]);
            s.keys[s.digit_local[d] + s.warp_cnt[warp][d] + rank[j]] = key[j];
        }
    }
    if constexpr (!std::is_same_v<Visit, NoVisit>) {   // after the ranking, whose registers are free again
#pragma unroll
        for (int j = 0; j < kSweepItems; ++j) {
            const uint32_t e = warp_base + j * 32 + lane;
            if (e < tile_count) visit(tile_base + e, key[j]);
        }
    }
    for (uint32_t d = threadIdx.x; d <= mask; d += kSweepThreads) {
        uint32_t excl = 0;
        if (tile > 0) {
            uint32_t p = tile - 1;
            uint32_t spins = 0;
            while (true) {
                const W w = SW::load(status + (size_t)p * kRadix + d);
                if ((w >> SW::kShift) == 0) {     // predecessor has not ranked its keys yet
                    if (++spins > (1u << 28)) __trap();
                    continue;
                }
                excl += (uint32_t)(w & SW::kValueMask);
                if (w & SW::kPrefix) break;        // tile 0 always publishes PREFIX: p never underflows
                --p;
            }
            SW::store(status + (size_t)tile * kRadix + d, SW::kPrefix | (W)(excl + s.digit_total[d]));
        }
        s.digit_global[d] = digit_base[d] + excl - s.digit_local[d];
    }
    __syncthreads();

    // contiguous runs out to global memory
    for (uint32_t i = threadIdx.x; i < tile_count; i += kSweepThreads) {
        const uint64_t k = s.keys[i];
        const uint32_t d = dg(k);
        store(out, (uint64_t)(s.digit_global[d] + i), k);
    }
}

template <typename W, typename Store = StoreKeys, typename Visit = NoVisit>
int sweep_pass(kombgpu_ctx *ctx, const uint64_t *src, uint64_t *dst, uint64_t n, const RadixPass &pass, const DigitSpec &dg,
               const uint32_t *digit_base, W *status, uint32_t *tile_counter, Store store = Store{}, Visit visit = Visit{}) {
    auto *kernel = pass.bits + pass.bits2 == 8 ? radix_sweep_kernel<W, 8, Store, Visit> : radix_sweep_kernel<W, 0, Store, Visit>;
    KG_LAUNCH(ctx, kernel, ceil_div_u64(n, kSweepTile), kSweepThreads, sizeof(SweepSmem), src, dst, n, dg, digit_base, status,
              tile_counter, store, visit);
    return KOMBGPU_OK;
}

// one pass: the key array or the CSR sink, with or without the first pass's visit
template <typename W>
int sweep_pass_opt(kombgpu_ctx *ctx, const uint64_t *src, uint64_t *dst, uint64_t n, const RadixPass &pass, const DigitSpec &dg,
                   const uint32_t *digit_base, W *status, uint32_t *tile_counter, bool to_col, bool visit, const SortOptions &o) {
    const StoreCol sc{o.col_base, o.col};
    const VisitFwdCol vf{o.fwd_row_ptr, o.col_base, o.col};
    if (to_col && visit) return sweep_pass(ctx, src, nullptr, n, pass, dg, digit_base, status, tile_counter, sc, vf);
    if (to_col) return sweep_pass(ctx, src, nullptr, n, pass, dg, digit_base, status, tile_counter, sc);
    if (visit) return sweep_pass(ctx, src, dst, n, pass, dg, digit_base, status, tile_counter, StoreKeys{}, vf);
    return sweep_pass(ctx, src, dst, n, pass, dg, digit_base, status, tile_counter);
}

// hist[p * 256 + d] += counts[x] for every x < m whose pass-p digit is d: the histograms of keys whose digits all lie in
// their low word, from the number of keys per low word (neighbouring x share their high digits: one atomic per warp)
__global__ void __launch_bounds__(kRsThreads) radix_count_hist_kernel(const uint32_t *__restrict__ counts, uint32_t m, PassList pl,
                                                                      uint32_t *__restrict__ hist) {
    __shared__ uint32_t s_hist[kMaxPasses * kRadix];
    for (int i = threadIdx.x; i < pl.n * kRadix; i += kRsThreads) s_hist[i] = 0;
    __syncthreads();
    const uint32_t lane = lane_id();
    for (uint64_t base = (uint64_t)blockIdx.x * kRsThreads; base < m; base += (uint64_t)gridDim.x * kRsThreads) {
        const uint64_t x = base + threadIdx.x;
        const uint32_t c = x < m ? counts[x] : 0u;
        for (int p = 0; p < pl.n; ++p) {
            const uint32_t d = pl.dg[p](x);
            const uint32_t d0 = __shfl_sync(kFullMask, d, 0);
            if (__all_sync(kFullMask, d == d0)) {
                const uint32_t sum = warp_reduce_add(c);
                if (lane == 0 && sum) atomicAdd(&s_hist[p * kRadix + d0], sum);
            } else if (c) {
                atomicAdd(&s_hist[p * kRadix + d], c);
            }
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < pl.n * kRadix; i += kRsThreads)
        if (s_hist[i]) atomicAdd(&hist[i], s_hist[i]);
}

// a sort without passes (fewer than 2 keys, or no digit bits): the keys are visited and go through the sink in their order
__global__ void store_unsorted_kernel(const uint64_t *__restrict__ keys, uint64_t n, StoreCol store, VisitFwdCol visit, bool do_visit) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        if (do_visit) visit(i, keys[i]);
        store(nullptr, i, keys[i]);
    }
}

template <typename Store, typename Visit>
int set_sweep_attrs(kombgpu_ctx *ctx) {
    KG_CUDA(ctx, cudaFuncSetAttribute(radix_sweep_kernel<uint32_t, 8, Store, Visit>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SweepSmem)));
    KG_CUDA(ctx, cudaFuncSetAttribute(radix_sweep_kernel<uint32_t, 0, Store, Visit>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SweepSmem)));
    KG_CUDA(ctx, cudaFuncSetAttribute(radix_sweep_kernel<uint64_t, 8, Store, Visit>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SweepSmem)));
    KG_CUDA(ctx, cudaFuncSetAttribute(radix_sweep_kernel<uint64_t, 0, Store, Visit>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SweepSmem)));
    return KOMBGPU_OK;
}

}  // namespace

int plan_radix_passes(int lo0, int hi0, int lo1, int hi1, RadixPass *out) {
    const int len0 = hi0 > lo0 ? hi0 - lo0 : 0, len1 = hi1 > lo1 ? hi1 - lo1 : 0;
    const int total = len0 + len1;
    if (total <= 0) return 0;
    const int np = (total + 7) / 8;
    const int w = (total + np - 1) / np;
    int n = 0;
    for (int v = 0; v < total; v += w) {            // virtual bits [v, e) of the concatenated ranges
        const int e = v + w < total ? v + w : total;
        RadixPass p{0, 0, 0, 0};
        if (e <= len0) { p.shift = lo0 + v; p.bits = e - v; }                       // inside the first range
        else if (v >= len0) { p.shift = lo1 + (v - len0); p.bits = e - v; }          // inside the second range
        else { p.shift = lo0 + v; p.bits = len0 - v; p.shift2 = lo1; p.bits2 = e - len0; }   // straddles the gap
        out[n++] = p;
    }
    return n;
}

int radix_sort_u64(kombgpu_ctx *ctx, uint64_t *a, uint64_t *b, uint64_t n, const RadixPass *passes, int n_passes,
                   uint64_t **sorted, const SortOptions *opt) {
    static const SortOptions kNone{};
    if (!opt) opt = &kNone;
    const bool to_col = opt->col != nullptr;
    const uint64_t *first = opt->first ? opt->first : a;
    *sorted = to_col ? nullptr : a;
    if (n < 2 || n_passes == 0) {
        if (to_col && n)
            KG_LAUNCH(ctx, store_unsorted_kernel, min(ceil_div_u64(n, 256), 148u * 16u), 256, 0, first, n, StoreCol{opt->col_base, opt->col},
                      VisitFwdCol{opt->fwd_row_ptr, opt->col_base, opt->col}, opt->fwd_row_ptr != nullptr);
        else if (opt->first && n)
            KG_CUDA(ctx, cudaMemcpyAsync(a, first, n * sizeof(uint64_t), cudaMemcpyDeviceToDevice, ctx->stream));
        return KOMBGPU_OK;
    }
    if (n >= (1ull << 32)) return ctx_fail(ctx, KOMBGPU_EINVAL, "radix_sort_u64: %llu keys exceed the 2^32 per-array limit", (unsigned long long)n);
    if (n_passes > kMaxPasses) return ctx_fail(ctx, KOMBGPU_EINVAL, "radix_sort_u64: %d passes exceed %d", n_passes, kMaxPasses);
    if (!ctx->sort_attr_set) {   // function attributes are per device: once per context, not per process
        KG_TRY((set_sweep_attrs<StoreKeys, NoVisit>(ctx)));
        KG_TRY((set_sweep_attrs<StoreCol, NoVisit>(ctx)));
        KG_TRY((set_sweep_attrs<StoreKeys, VisitFwdCol>(ctx)));
        KG_TRY((set_sweep_attrs<StoreCol, VisitFwdCol>(ctx)));
        ctx->sort_attr_set = true;
    }
    // Workspace, in 32-bit words: [n_passes x 256 digit histograms | kMaxPasses tile counters | status words].  Below 2^30
    // keys every pass has its own region of 32-bit words, all zeroed at once.  From 2^30 on the passes share one region
    // of 64-bit words (n/4 bytes), zeroed again before each pass: one region per pass would cost up to 8 GiB.  The head
    // has an even number of words, so the 64-bit words stay aligned.
    const bool wide = n >= (1ull << 30);
    const size_t region = (size_t)ceil_div_u64(n, kSweepTile) * kRadix;   // status words of one pass
    const size_t head = (size_t)n_passes * kRadix + kMaxPasses;
    const size_t words = head + (wide ? 2 * region : (size_t)n_passes * region);
    DevBuf<uint32_t> ws;
    KG_ALLOC(ctx, ws, words);
    KG_CUDA(ctx, cudaMemsetAsync(ws.p, 0, words * sizeof(uint32_t), ctx->stream));
    PassList pl{};
    pl.n = n_passes;
    for (int p = 0; p < n_passes; ++p) pl.dg[p] = DigitSpec::of(passes[p]);
    if (opt->counts) {
        const uint32_t m = opt->n_counts;
        if (m) KG_LAUNCH(ctx, radix_count_hist_kernel, min(ceil_div_u64(m, kRsThreads), (uint32_t)ctx->sm_count * 4u), kRsThreads, 0,
                         opt->counts, m, pl, ws.p);
    } else {
        const uint32_t hist_grid = min(ceil_div_u64(n, kRsTile), (uint32_t)ctx->sm_count * 4u);
        KG_LAUNCH(ctx, radix_global_hist_kernel, hist_grid, kRsThreads, 0, first, n, pl, ws.p);
    }
    KG_LAUNCH(ctx, radix_hist_scan_kernel, n_passes, kRadix, 0, ws.p);
    // ping-pong: pass 0 reads `first` (a, or the caller's const keys) and writes b; later passes alternate b and a
    const uint64_t *src = first;
    uint64_t *dst = b;
    for (int p = 0; p < n_passes; ++p) {
        const uint32_t *digit_base = ws.p + (size_t)p * kRadix;
        uint32_t *counter = ws.p + (size_t)n_passes * kRadix + p;
        uint64_t *status64 = reinterpret_cast<uint64_t *>(ws.p + head);
        uint32_t *status32 = ws.p + head + (size_t)p * region;
        if (wide && p > 0) KG_CUDA(ctx, cudaMemsetAsync(status64, 0, region * sizeof(uint64_t), ctx->stream));
        const bool last_to_col = to_col && p == n_passes - 1, visit = p == 0 && opt->fwd_row_ptr;
        if (wide) KG_TRY(sweep_pass_opt(ctx, src, dst, n, passes[p], pl.dg[p], digit_base, status64, counter, last_to_col, visit, *opt));
        else KG_TRY(sweep_pass_opt(ctx, src, dst, n, passes[p], pl.dg[p], digit_base, status32, counter, last_to_col, visit, *opt));
        if (last_to_col) break;
        *sorted = dst;
        src = dst;
        dst = dst == b ? a : b;
    }
    return KOMBGPU_OK;
}


namespace {

__device__ __forceinline__ uint64_t mix64(uint64_t x) {
    x ^= x >> 33; x *= 0xff51afd7ed558ccdull; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ull; x ^= x >> 33;
    return x;
}
__global__ void debug_fill_kernel(uint64_t *keys, uint64_t n, uint64_t lo_mask, uint64_t hi_mask, int sorted_hi) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t h = mix64(i + 0x9e3779b97f4a7c15ull);
        const uint64_t hi = sorted_hi ? ((i * (hi_mask + 1)) / n) : ((h >> 32) & hi_mask);
        keys[i] = (hi << 32) | (h & lo_mask);
    }
}
// out[0] += sum of keys, out[1] ^= mix of keys, out[2] += number of descents
__global__ void debug_check_kernel(const uint64_t *keys, uint64_t n, unsigned long long *out) {
    unsigned long long sum = 0, x = 0, bad = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        sum += keys[i];
        x ^= mix64(keys[i]);
        if (i && keys[i - 1] > keys[i]) ++bad;
    }
    atomicAdd(&out[0], sum);
    atomicXor(&out[1], x);
    if (bad) atomicAdd(&out[2], bad);
}

}  // namespace

}  // namespace kg

extern "C" int kombgpu_debug_sort_u64(kombgpu_ctx *ctx, uint64_t n, int lo_bits, int hi_bits, int sorted_hi, int reps,
                                      float *ms_best, int *ok) {
    using namespace kg;
    if (!ctx || !ms_best || !ok || n == 0 || lo_bits < 0 || lo_bits > 32 || hi_bits < 0 || hi_bits > 32 || reps < 1)
        return KOMBGPU_EINVAL;
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    DevBuf<uint64_t> src, a, b;
    DevBuf<unsigned long long> chk;
    KG_ALLOC(ctx, src, n);
    KG_ALLOC(ctx, a, n);
    KG_ALLOC(ctx, b, n);
    KG_ALLOC(ctx, chk, 6);
    KG_CUDA(ctx, cudaMemsetAsync(chk.p, 0, 6 * sizeof(unsigned long long), ctx->stream));
    const uint64_t lo_mask = lo_bits == 32 ? 0xffffffffull : ((1ull << lo_bits) - 1), hi_mask = hi_bits == 32 ? 0xffffffffull : ((1ull << hi_bits) - 1);
    const int grid = ctx->sm_count * 8;
    KG_LAUNCH(ctx, debug_fill_kernel, grid, 256, 0, src.p, n, lo_mask, hi_mask, sorted_hi);
    KG_LAUNCH(ctx, debug_check_kernel, grid, 256, 0, src.p, n, chk.p);
    RadixPass passes[8];
    const int np = plan_radix_passes(0, lo_bits, 32, 32 + hi_bits, passes);
    float best = 1e30f;
    uint64_t *sorted = nullptr;
    cudaEvent_t e0, e1;
    KG_CUDA(ctx, cudaEventCreate(&e0));
    KG_CUDA(ctx, cudaEventCreate(&e1));
    for (int r = 0; r < reps; ++r) {
        KG_CUDA(ctx, cudaMemcpyAsync(a.p, src.p, n * sizeof(uint64_t), cudaMemcpyDeviceToDevice, ctx->stream));
        KG_CUDA(ctx, cudaEventRecord(e0, ctx->stream));
        int rc = radix_sort_u64(ctx, a.p, b.p, n, passes, np, &sorted);
        if (rc != KOMBGPU_OK) return rc;
        KG_CUDA(ctx, cudaEventRecord(e1, ctx->stream));
        KG_CUDA(ctx, cudaEventSynchronize(e1));
        float ms = 0;
        KG_CUDA(ctx, cudaEventElapsedTime(&ms, e0, e1));
        if (ms < best) best = ms;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    KG_LAUNCH(ctx, debug_check_kernel, grid, 256, 0, sorted, n, chk.p + 3);
    unsigned long long h[6];
    KG_TRY(read_back(ctx, chk.p, h, 6));
    *ok = (h[0] == h[3] && h[1] == h[4] && h[5] == 0) ? 1 : 0;   // same multiset (sum + xor of mixes), no descent
    *ms_best = best;
    return KOMBGPU_OK;
}
