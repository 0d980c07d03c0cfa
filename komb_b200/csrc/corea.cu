// corea.cu — stage 3: CORE-A anomaly score.
//
// Restates CoreA::getAnomalyScore / fractionalRank (src/CoreA.h:109-187):
//   key_i   = coreness_i * n + degree_i            (int32 wrap = "ref32", quirk Q5; int64 = "exact64")
//   a_i     = descending average-tie rank of degree_i
//   b_i     = descending average-tie rank of key_i
//   score_i = | ln a_i - ln b_i |
// The reference ranks in O(n * distinct values); here
//   degree ranks: histogram over [0, max degree] -> prefix scan -> rank LUT
//   key ranks   : radix sort of (key << 32 | vertex) -> run boundaries -> rank
// exact64 keys are ranked as the pair (coreness + degree / n, degree % n), which
// orders exactly like coreness * n + degree, also for degrees >= n.
// Ranks are exact half-integers in FP64 (class [s, e) of the ascending order has
// descending average rank n - (s + e - 1) / 2); only ln() can differ from glibc,
// by <= 1 ulp: the scores are held to 6e-14 absolute of the exact ranks' logs.
#include <cstdlib>
#include <cstring>

#include "dgraph.cuh"
#include "primitives.cuh"

namespace kg {

namespace {

constexpr int kThreads = 256;
constexpr int kSmemBins = 4096;

inline uint32_t grid_for(uint64_t n, int per_block, uint32_t cap) {
    uint32_t g = ceil_div_u64(n ? n : 1, per_block);
    return g < cap ? g : cap;
}

// exact64 key coreness * n + degree as the pair (high, low) = (coreness + degree / n, degree % n): the degree's
// multiples of n carried into the coreness, so the pair orders exactly like the int64 key even for degrees >= n
__device__ __forceinline__ uint2 exact_pair(int32_t core, int32_t deg, uint32_t n) {
    uint32_t c = (uint32_t)core, d = (uint32_t)deg;
    if (d >= n) { c += d / n; d %= n; }
    return make_uint2(c, d);
}
// bit widths of the two fields of exact_pair over coreness <= max_core, degree <= max_deg (n >= 1)
inline void exact_pair_bits(uint32_t max_core, uint32_t max_deg, uint32_t n, int *core_bits, int *deg_bits) {
    *core_bits = bits_for((uint64_t)max_core + max_deg / n);
    *deg_bits = bits_for(max_deg < n ? max_deg : n - 1);
}

// mm[0] = max degree, mm[1] = max coreness, mm[2] = 1 if any value is negative (input validation)
__global__ void __launch_bounds__(kThreads) max2_kernel(const int32_t *__restrict__ deg, const int32_t *__restrict__ core,
                                                        uint32_t n, int32_t *__restrict__ mm) {
    int32_t md = 0, mc = 0, lo = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const int32_t d = deg[i], c = core[i];
        md = max(md, d);
        mc = max(mc, c);
        lo = min(lo, min(d, c));
    }
    md = warp_reduce_max(md);
    mc = warp_reduce_max(mc);
    lo = warp_reduce_min(lo);
    if (lane_id() == 0) {
        if (md) atomicMax(&mm[0], md);
        if (mc) atomicMax(&mm[1], mc);
        if (lo < 0) atomicExch(&mm[2], 1);
    }
}

// degree histogram: low degrees (the bulk of a power-law graph) are counted in a
// per-CTA shared-memory histogram, the tail goes straight to global atomics.
__global__ void __launch_bounds__(kThreads) degree_hist_kernel(const int32_t *__restrict__ deg, uint32_t n,
                                                               uint32_t n_bins, uint32_t *__restrict__ hist) {
    __shared__ uint32_t s_hist[kSmemBins];
    for (int b = threadIdx.x; b < kSmemBins; b += kThreads) s_hist[b] = 0;
    __syncthreads();
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t d = (uint32_t)deg[i];
        if (d < kSmemBins) atomicAdd(&s_hist[d], 1u);
        else atomicAdd(&hist[d], 1u);
    }
    __syncthreads();
    for (uint32_t b = threadIdx.x; b < kSmemBins && b < n_bins; b += kThreads) {
        uint32_t c = s_hist[b];
        if (c) atomicAdd(&hist[b], c);
    }
}

// rank_lut[d] = #{degree > d} + (count(d) + 1) / 2
struct HistIn {
    const uint32_t *hist;
    __device__ uint32_t operator()(uint64_t d) const { return hist[d]; }
};
struct RankLutOut {
    double *lut;
    uint32_t n;
    __device__ void operator()(uint64_t d, uint32_t less, uint32_t cnt) const {
        uint32_t greater = n - less - cnt;
        lut[d] = (double)greater + 0.5 * (double)(cnt + 1u);
    }
};

// sort key: high word orders the vertices by CORE-A key, low word = vertex id
// (`count` elements; `n` is the vertex count of the WHOLE graph, which enters the reference's key arithmetic)
__global__ void __launch_bounds__(kThreads) pack_rank_keys_kernel(const int32_t *__restrict__ core,
                                                                  const int32_t *__restrict__ deg, uint32_t count, uint32_t n, int mode,
                                                                  int deg_bits, uint64_t *__restrict__ keys) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t hi;
        if (mode == 0) {
            // (int32)(coreness * n + degree) with two's complement wrap; flip the sign bit for unsigned order
            hi = ((uint32_t)core[i] * n + (uint32_t)deg[i]) ^ 0x80000000u;
        } else if (mode == 1) {
            const uint2 p = exact_pair(core[i], deg[i], n);
            hi = (p.x << deg_bits) | p.y;
        } else if (mode == 2) {
            hi = exact_pair(core[i], deg[i], n).y;   // wide fallback, first sort: by the low field
        } else {
            hi = 0;
        }
        keys[i] = ((uint64_t)hi << 32) | (uint32_t)i;
    }
}

// wide fallback, second sort: re-key the sequence sorted by the low field by the high field
// (`count` keys; `n` is the vertex count of the whole graph)
__global__ void __launch_bounds__(kThreads) rekey_by_core_kernel(const int32_t *__restrict__ core, const int32_t *__restrict__ deg,
                                                                 uint32_t count, uint32_t n, uint64_t *__restrict__ keys) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t v = (uint32_t)keys[i];
        keys[i] = ((uint64_t)exact_pair(core[v], deg[v], n).x << 32) | v;
    }
}

// class heads of the sorted sequence.  wide = compare the exact64 pairs through
// the vertex id instead of the packed high word.
struct ClassFlagIn {
    const uint64_t *keys;
    const int32_t *core;
    const int32_t *deg;
    uint32_t n;
    int wide;
    __device__ uint32_t operator()(uint64_t i) const {
        if (i == 0) return 1u;
        if (!wide) return (keys[i] >> 32) != (keys[i - 1] >> 32) ? 1u : 0u;
        uint32_t a = (uint32_t)keys[i], b = (uint32_t)keys[i - 1];
        const uint2 pa = exact_pair(core[a], deg[a], n), pb = exact_pair(core[b], deg[b], n);
        return (pa.x != pb.x || pa.y != pb.y) ? 1u : 0u;
    }
};
struct ClassFlagOut {
    uint32_t *head_pos;  // [n_classes] start position of each class
    uint32_t *cls;       // [n] class of each sorted position
    __device__ void operator()(uint64_t i, uint32_t prefix, uint32_t flag) const {
        if (flag) head_pos[prefix] = (uint32_t)i;
        cls[i] = prefix + flag - 1u;
    }
};

__global__ void __launch_bounds__(kThreads) score_kernel(const uint64_t *__restrict__ keys, const uint32_t *__restrict__ cls,
                                                         const uint32_t *__restrict__ head_pos,
                                                         const uint32_t *__restrict__ n_classes_dev,
                                                         const int32_t *__restrict__ deg, const double *__restrict__ deg_lut,
                                                         uint32_t n, double *__restrict__ score,
                                                         unsigned long long *__restrict__ max_bits) {
    const uint32_t n_classes = *n_classes_dev;
    double local_max = 0.0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t c = cls[i];
        const uint32_t s = head_pos[c];
        const uint32_t e = c + 1 < n_classes ? head_pos[c + 1] : n;
        // ascending positions [s, e)  ->  descending ranks n-e+1 .. n-s, mean n - (s+e-1)/2
        const double key_rank = (double)n - 0.5 * (double)((uint64_t)s + e - 1);
        const uint32_t v = (uint32_t)keys[i];
        const double deg_rank = deg_lut[deg[v]];
        const double sc = fabs(log(deg_rank) - log(key_rank));
        score[v] = sc;
        local_max = fmax(local_max, sc);
    }
    // scores are >= 0, so their bit patterns order like unsigned integers
    unsigned long long bits = (unsigned long long)__double_as_longlong(local_max);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        unsigned long long t = __shfl_xor_sync(kFullMask, bits, o);
        bits = t > bits ? t : bits;
    }
    if (lane_id() == 0 && bits) atomicMax(max_bits, bits);
}

// ---- small key spaces: no sort at all.  When (max coreness + 1) x (max degree + 1) is small (the usual unitig graph:
// a few dozen coreness levels, a few hundred degrees) the (coreness, degree) pairs are counted in a 2-D histogram;
// while no degree reaches n and (ref32) nothing wraps, the key coreness * n + degree orders like the pair, so the key
// ranks are a prefix scan over the bins (the same LUT trick as the degree ranks, whose histogram is the bins' column sums).
constexpr uint32_t kPairBinsSmem = 12288;        // 48 KB of shared-memory counters
constexpr uint64_t kPairBinsMax = 1ull << 22;    // above this the sort-based path is used

__global__ void __launch_bounds__(kThreads) pair_hist_kernel(const int32_t *__restrict__ core, const int32_t *__restrict__ deg, uint32_t n,
                                                             uint32_t n_deg, uint32_t n_bins, uint32_t *__restrict__ hist) {
    extern __shared__ uint32_t s_pair[];
    const bool use_smem = n_bins <= kPairBinsSmem;
    if (use_smem) {
        for (uint32_t b = threadIdx.x; b < n_bins; b += kThreads) s_pair[b] = 0;
        __syncthreads();
    }
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t b = (uint32_t)core[i] * n_deg + (uint32_t)deg[i];
        if (use_smem) atomicAdd(&s_pair[b], 1u);
        else atomicAdd(&hist[b], 1u);
    }
    if (use_smem) {
        __syncthreads();
        for (uint32_t b = threadIdx.x; b < n_bins; b += kThreads) {
            const uint32_t c = s_pair[b];
            if (c) atomicAdd(&hist[b], c);
        }
    }
}
// degree histogram = column sums of the pair histogram
__global__ void __launch_bounds__(kThreads) pair_hist_columns_kernel(const uint32_t *__restrict__ pair, uint32_t n_core, uint32_t n_deg,
                                                                     uint32_t *__restrict__ deg_hist) {
    for (uint32_t d = blockIdx.x * blockDim.x + threadIdx.x; d < n_deg; d += gridDim.x * blockDim.x) {
        uint32_t s = 0;
        for (uint32_t c = 0; c < n_core; ++c) s += pair[(uint64_t)c * n_deg + d];
        deg_hist[d] = s;
    }
}
__global__ void __launch_bounds__(kThreads) score_lut_kernel(const int32_t *__restrict__ core, const int32_t *__restrict__ deg, uint32_t n,
                                                             uint32_t n_deg, const double *__restrict__ deg_lut,
                                                             const double *__restrict__ key_lut, double *__restrict__ score,
                                                             unsigned long long *__restrict__ max_bits) {
    double local_max = 0.0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t d = (uint32_t)deg[i];
        const double sc = fabs(log(deg_lut[d]) - log(key_lut[(uint64_t)(uint32_t)core[i] * n_deg + d]));
        score[i] = sc;
        local_max = fmax(local_max, sc);
    }
    unsigned long long bits = (unsigned long long)__double_as_longlong(local_max);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        unsigned long long t = __shfl_xor_sync(kFullMask, bits, o);
        bits = t > bits ? t : bits;
    }
    if (lane_id() == 0 && bits) atomicMax(max_bits, bits);
}

}  // namespace

int corea_scores(kombgpu_ctx *ctx, const int32_t *core, const int32_t *deg, uint32_t n, int key_mode, double *score,
                 double *max_score_host) {
    *max_score_host = 0.0;
    if (n == 0) return KOMBGPU_OK;
    if (key_mode != KOMBGPU_KEY_REF32 && key_mode != KOMBGPU_KEY_EXACT64)
        return ctx_fail(ctx, KOMBGPU_EINVAL, "unknown CORE-A key mode %d", key_mode);
    const uint32_t cap = (uint32_t)ctx->sm_count * 8u;

    DevBuf<int32_t> mm(ctx, 3);
    if (!mm) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
    KG_CUDA(ctx, cudaMemsetAsync(mm.p, 0, 3 * sizeof(int32_t), ctx->stream));
    KG_LAUNCH(ctx, max2_kernel, grid_for(n, kThreads, cap), kThreads, 0, deg, core, n, mm.p);
    int32_t h_mm[3] = {0, 0, 0};
    KG_TRY(read_back(ctx, mm.p, h_mm, 3));
    if (h_mm[2]) return ctx_fail(ctx, KOMBGPU_EINVAL, "negative coreness or degree");
    const uint32_t max_deg = (uint32_t)h_mm[0], max_core = (uint32_t)h_mm[1];

    // small key space: ranks from the 2-D histogram, no sort.  The keys order like the raw pair (coreness, degree) only
    // while no degree >= n carries into the coreness and, for ref32, coreness * n + degree does not wrap.
    const uint64_t n_pair_bins = (uint64_t)(max_core + 1) * (uint64_t)(max_deg + 1);
    const bool pair_order = max_deg < n && (key_mode == KOMBGPU_KEY_EXACT64 || (uint64_t)max_core * n + max_deg <= 0x7fffffffull);
    const bool no_lut = getenv("KOMBGPU_COREA_SORT") != nullptr;   // A/B runs and tests: force the sort-based path
    if (n_pair_bins <= kPairBinsMax && pair_order && !no_lut) {
        const uint32_t n_deg = max_deg + 1, n_core = max_core + 1, nb = (uint32_t)n_pair_bins;
        DevBuf<uint32_t> pair, dh;
        DevBuf<double> key_lut, deg_lut;
        DevBuf<unsigned long long> max_bits(ctx, 1);
        KG_ALLOC(ctx, pair, nb);
        KG_ALLOC(ctx, dh, n_deg);
        KG_ALLOC(ctx, key_lut, nb);
        KG_ALLOC(ctx, deg_lut, n_deg);
        if (!max_bits) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
        KG_CUDA(ctx, cudaMemsetAsync(pair.p, 0, (size_t)nb * sizeof(uint32_t), ctx->stream));
        KG_CUDA(ctx, cudaMemsetAsync(max_bits.p, 0, sizeof(unsigned long long), ctx->stream));
        if (!ctx->corea_attr_set) {
            KG_CUDA(ctx, cudaFuncSetAttribute(pair_hist_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kPairBinsSmem * sizeof(uint32_t))));
            ctx->corea_attr_set = true;
        }
        const size_t smem = nb <= kPairBinsSmem ? (size_t)nb * sizeof(uint32_t) : 0;
        KG_LAUNCH(ctx, pair_hist_kernel, grid_for(n, kThreads * 8, (uint32_t)ctx->sm_count * 2u), kThreads, smem, core, deg, n, n_deg, nb, pair.p);
        KG_LAUNCH(ctx, pair_hist_columns_kernel, grid_for(n_deg, kThreads, cap), kThreads, 0, pair.p, n_core, n_deg, dh.p);
        KG_TRY((device_scan<uint32_t>(ctx, n_deg, HistIn{dh.p}, RankLutOut{deg_lut.p, n}, (uint32_t *)nullptr)));
        KG_TRY((device_scan<uint32_t>(ctx, nb, HistIn{pair.p}, RankLutOut{key_lut.p, n}, (uint32_t *)nullptr)));
        KG_LAUNCH(ctx, score_lut_kernel, grid_for(n, kThreads, cap), kThreads, 0, core, deg, n, n_deg, deg_lut.p, key_lut.p, score, max_bits.p);
        unsigned long long h_bits = 0;
        KG_TRY(read_back(ctx, max_bits.p, &h_bits, 1));
        memcpy(max_score_host, &h_bits, sizeof(double));
        return KOMBGPU_OK;
    }

    // degree ranks through a histogram LUT
    const uint32_t n_bins = max_deg + 1;
    DevBuf<uint32_t> hist;
    DevBuf<double> lut;
    KG_ALLOC(ctx, hist, n_bins);
    KG_ALLOC(ctx, lut, n_bins);
    KG_CUDA(ctx, cudaMemsetAsync(hist.p, 0, (size_t)n_bins * sizeof(uint32_t), ctx->stream));
    KG_LAUNCH(ctx, degree_hist_kernel, grid_for(n, kThreads * 8, cap), kThreads, 0, deg, n, n_bins, hist.p);
    KG_TRY((device_scan<uint32_t>(ctx, n_bins, HistIn{hist.p}, RankLutOut{lut.p, n}, (uint32_t *)nullptr)));

    // key ranks through a sort
    DevBuf<uint64_t> ka, kb;
    KG_ALLOC(ctx, ka, n);
    KG_ALLOC(ctx, kb, n);
    uint64_t *sorted = ka.p;
    RadixPass passes[8];
    int wide = 0;
    if (key_mode == KOMBGPU_KEY_REF32) {
        KG_LAUNCH(ctx, pack_rank_keys_kernel, grid_for(n, kThreads, cap), kThreads, 0, core, deg, n, n, 0, 0, ka.p);
        int np = plan_radix_passes(32, 64, 0, 0, passes);
        KG_TRY(radix_sort_u64(ctx, ka.p, kb.p, n, passes, np, &sorted));
    } else {
        int cb, db;
        exact_pair_bits(max_core, max_deg, n, &cb, &db);
        if (db + cb <= 32) {
            KG_LAUNCH(ctx, pack_rank_keys_kernel, grid_for(n, kThreads, cap), kThreads, 0, core, deg, n, n, 1, db, ka.p);
            int np = plan_radix_passes(32, 32 + db + cb, 0, 0, passes);
            KG_TRY(radix_sort_u64(ctx, ka.p, kb.p, n, passes, np, &sorted));
        } else {
            // the pair does not fit 32 bits: LSD over its two fields with a re-key in between
            wide = 1;
            KG_LAUNCH(ctx, pack_rank_keys_kernel, grid_for(n, kThreads, cap), kThreads, 0, core, deg, n, n, 2, 0, ka.p);
            int np = plan_radix_passes(32, 32 + db, 0, 0, passes);
            KG_TRY(radix_sort_u64(ctx, ka.p, kb.p, n, passes, np, &sorted));
            uint64_t *other = sorted == ka.p ? kb.p : ka.p;
            KG_LAUNCH(ctx, rekey_by_core_kernel, grid_for(n, kThreads, cap), kThreads, 0, core, deg, n, n, sorted);
            np = plan_radix_passes(32, 32 + cb, 0, 0, passes);
            uint64_t *sorted2 = sorted;
            KG_TRY(radix_sort_u64(ctx, sorted, other, n, passes, np, &sorted2));
            sorted = sorted2;
        }
    }

    DevBuf<uint32_t> head_pos, cls, n_classes(ctx, 1);
    DevBuf<unsigned long long> max_bits(ctx, 1);
    KG_ALLOC(ctx, head_pos, n);
    KG_ALLOC(ctx, cls, n);
    if (!n_classes || !max_bits) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
    KG_CUDA(ctx, cudaMemsetAsync(max_bits.p, 0, sizeof(unsigned long long), ctx->stream));
    KG_TRY((device_scan<uint32_t>(ctx, n, ClassFlagIn{sorted, core, deg, n, wide}, ClassFlagOut{head_pos.p, cls.p}, n_classes.p)));
    KG_LAUNCH(ctx, score_kernel, grid_for(n, kThreads, cap), kThreads, 0, sorted, cls.p, head_pos.p, n_classes.p, deg, lut.p, n,
              score, max_bits.p);
    unsigned long long h_bits = 0;
    KG_TRY(read_back(ctx, max_bits.p, &h_bits, 1));
    memcpy(max_score_host, &h_bits, sizeof(double));
    return KOMBGPU_OK;
}


// ---------------------------------------------------------------------------------------------------------------
// CORE-A over the ranks of a communicator (SURVEY.md section 8(e), row 4): every rank scores its own unitigs.
//   degree ranks   the degree histograms of all ranks are summed (each rank reads its peers' histograms from
//                  peer memory), then the same prefix scan -> LUT as on one GPU
//   key ranks      a rank sorts ITS keys and turns them into a list of distinct keys with their first positions;
//                  the global rank of a key class is n - (2 * less + equal - 1) / 2 with less / equal summed over
//                  the ranks' lists by binary search -- the lists are tiny next to the vertex arrays (distinct
//                  (coreness, degree) pairs), so nothing of size n ever crosses a link
// Ranks are exact half-integers as before; the result does not depend on the partition.
// ---------------------------------------------------------------------------------------------------------------
namespace {

__global__ void __launch_bounds__(kThreads) sum_peer_hist_kernel(PeerPtrs<uint32_t> hist, int world, uint32_t n_bins,
                                                                 uint32_t *__restrict__ total) {
    for (uint64_t d = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; d < n_bins; d += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t s = 0;
        for (int q = 0; q < world; ++q) s += hist.p[q][d];
        total[d] = s;
    }
}

// distinct key of every class of the locally sorted sequence, as a 64-bit value that orders like the sort did
__global__ void __launch_bounds__(kThreads) class_keys_kernel(const uint64_t *__restrict__ sorted, const uint32_t *__restrict__ head_pos,
                                                              uint32_t n_classes, const int32_t *__restrict__ core,
                                                              const int32_t *__restrict__ deg, uint32_t n_global, int key_mode,
                                                              uint64_t *__restrict__ dkey, uint32_t *__restrict__ dhead) {
    for (uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; c < n_classes; c += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t h = head_pos[c];
        const uint32_t v = (uint32_t)sorted[h];
        if (key_mode == KOMBGPU_KEY_REF32) {
            dkey[c] = (uint64_t)(((uint32_t)core[v] * n_global + (uint32_t)deg[v]) ^ 0x80000000u);
        } else {
            const uint2 p = exact_pair(core[v], deg[v], n_global);
            dkey[c] = ((uint64_t)p.x << 32) | p.y;
        }
        dhead[c] = h;
    }
}

struct ClassLists {
    const uint64_t *key[kMaxRanks];
    const uint32_t *head[kMaxRanks];
    uint32_t n_classes[kMaxRanks];
    uint32_t n_local[kMaxRanks];
};

// global descending average rank of every local class
__global__ void __launch_bounds__(kThreads) class_rank_kernel(ClassLists L, int world, int rank, uint32_t n_global,
                                                              double *__restrict__ class_rank) {
    const uint32_t n_mine = L.n_classes[rank];
    for (uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; c < n_mine; c += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t x = L.key[rank][c];
        uint64_t less = 0, eq = 0;
        for (int q = 0; q < world; ++q) {
            const uint32_t dq = L.n_classes[q];
            uint32_t lo = 0, hi = dq;   // first class of rank q whose key is >= x
            while (lo < hi) {
                const uint32_t mid = (lo + hi) >> 1;
                if (L.key[q][mid] < x) lo = mid + 1; else hi = mid;
            }
            const uint32_t at = lo < dq ? L.head[q][lo] : L.n_local[q];
            less += at;
            if (lo < dq && L.key[q][lo] == x) eq += (lo + 1 < dq ? L.head[q][lo + 1] : L.n_local[q]) - at;
        }
        // ascending positions [less, less + eq) of the global order -> descending ranks, mean n - (2 less + eq - 1) / 2
        class_rank[c] = (double)n_global - 0.5 * (double)(2 * less + eq - 1);
    }
}

__global__ void __launch_bounds__(kThreads) dist_score_kernel(const uint64_t *__restrict__ sorted, const uint32_t *__restrict__ cls,
                                                              const double *__restrict__ class_rank, const int32_t *__restrict__ deg,
                                                              const double *__restrict__ deg_lut, uint32_t n_local,
                                                              double *__restrict__ score, unsigned long long *__restrict__ max_bits) {
    double local_max = 0.0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_local; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t v = (uint32_t)sorted[i];
        const double sc = fabs(log(deg_lut[deg[v]]) - log(class_rank[cls[i]]));
        score[v] = sc;
        local_max = fmax(local_max, sc);
    }
    unsigned long long bits = (unsigned long long)__double_as_longlong(local_max);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        unsigned long long t = __shfl_xor_sync(kFullMask, bits, o);
        bits = t > bits ? t : bits;
    }
    if (lane_id() == 0 && bits) atomicMax(max_bits, bits);
}

}  // namespace

int dist_corea(kombgpu_dist_graph *g, int key_mode) {
    kombgpu_comm *c = g->comm;
    kombgpu_ctx *ctx = g->ctx;
    const int world = c->world;
    const uint32_t n_local = g->n_local, n = g->n_global;
    if (key_mode != KOMBGPU_KEY_REF32 && key_mode != KOMBGPU_KEY_EXACT64)
        return ctx_fail(ctx, KOMBGPU_EINVAL, "unknown CORE-A key mode %d", key_mode);
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    KG_CUDA(ctx, cudaEventCreate(&ev0));
    KG_CUDA(ctx, cudaEventCreate(&ev1));
    KG_CUDA(ctx, cudaEventRecord(ev0, ctx->stream));
    if (!g->score) {
        g->score = static_cast<double *>(ws_alloc(ctx, (n_local ? n_local : 1) * sizeof(double)));
        if (!g->score) return ctx_fail(ctx, KOMBGPU_ENOMEM, "score array");
    }
    const uint32_t cap = (uint32_t)ctx->sm_count * 8u;
    const uint32_t max_deg = (uint32_t)g->st.max_degree, max_core = (uint32_t)(g->st.max_coreness > 0 ? g->st.max_coreness : 0);
    const SymMark mark = sym_mark(c);

    // ---- degree ranks: sum of the ranks' histograms -> LUT
    const uint32_t n_bins = max_deg + 1;
    uint32_t *hist = nullptr;
    PeerPtrs<uint32_t> hist_peers{};
    KG_TRY(sym_alloc(c, (size_t)n_bins, &hist, &hist_peers));
    KG_CUDA(ctx, cudaMemsetAsync(hist, 0, (size_t)n_bins * sizeof(uint32_t), ctx->stream));
    if (n_local) KG_LAUNCH(ctx, degree_hist_kernel, grid_for(n_local, kThreads * 8, cap), kThreads, 0, g->deg, n_local, n_bins, hist);

    // ---- local key order (same kernels as the single-GPU path, keys built with the GLOBAL n)
    DevBuf<uint64_t> ka, kb;
    KG_ALLOC(ctx, ka, n_local);
    KG_ALLOC(ctx, kb, n_local);
    uint64_t *sorted = ka.p;
    RadixPass passes[8];
    int wide = 0;
    if (n_local) {
        if (key_mode == KOMBGPU_KEY_REF32) {
            KG_LAUNCH(ctx, pack_rank_keys_kernel, grid_for(n_local, kThreads, cap), kThreads, 0, g->core, g->deg, n_local, n, 0, 0, ka.p);
            int np = plan_radix_passes(32, 64, 0, 0, passes);
            KG_TRY(radix_sort_u64(ctx, ka.p, kb.p, n_local, passes, np, &sorted));
        } else {
            int cb, db;
            exact_pair_bits(max_core, max_deg, n, &cb, &db);
            if (db + cb <= 32) {
                KG_LAUNCH(ctx, pack_rank_keys_kernel, grid_for(n_local, kThreads, cap), kThreads, 0, g->core, g->deg, n_local, n, 1, db, ka.p);
                int np = plan_radix_passes(32, 32 + db + cb, 0, 0, passes);
                KG_TRY(radix_sort_u64(ctx, ka.p, kb.p, n_local, passes, np, &sorted));
            } else {
                wide = 1;
                KG_LAUNCH(ctx, pack_rank_keys_kernel, grid_for(n_local, kThreads, cap), kThreads, 0, g->core, g->deg, n_local, n, 2, 0, ka.p);
                int np = plan_radix_passes(32, 32 + db, 0, 0, passes);
                KG_TRY(radix_sort_u64(ctx, ka.p, kb.p, n_local, passes, np, &sorted));
                uint64_t *other = sorted == ka.p ? kb.p : ka.p;
                KG_LAUNCH(ctx, rekey_by_core_kernel, grid_for(n_local, kThreads, cap), kThreads, 0, g->core, g->deg, n_local, n, sorted);
                np = plan_radix_passes(32, 32 + cb, 0, 0, passes);
                uint64_t *sorted2 = sorted;
                KG_TRY(radix_sort_u64(ctx, sorted, other, n_local, passes, np, &sorted2));
                sorted = sorted2;
            }
        }
    }
    DevBuf<uint32_t> head_pos, cls, d_classes(ctx, 1);
    KG_ALLOC(ctx, head_pos, n_local);
    KG_ALLOC(ctx, cls, n_local);
    if (!d_classes) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
    KG_TRY((device_scan<uint32_t>(ctx, n_local, ClassFlagIn{sorted, g->core, g->deg, n, wide}, ClassFlagOut{head_pos.p, cls.p}, d_classes.p)));
    uint32_t n_classes = 0;
    KG_TRY(read_back(ctx, d_classes.p, &n_classes, 1));

    // ---- publish the list of distinct keys; meet; rank the local classes against every rank's list
    unsigned long long mine[2] = {n_classes, n_local}, all[kMaxRanks * 2];
    KG_TRY(comm_exchange(c, mine, 2, all));   // also: every rank's histogram is complete
    uint32_t max_classes = 1;
    ClassLists L{};
    for (int q = 0; q < world; ++q) {
        L.n_classes[q] = (uint32_t)all[q * 2];
        L.n_local[q] = (uint32_t)all[q * 2 + 1];
        if (L.n_classes[q] > max_classes) max_classes = L.n_classes[q];
    }
    uint64_t *dkey = nullptr;
    uint32_t *dhead = nullptr;
    PeerPtrs<uint64_t> dkey_peers{};
    PeerPtrs<uint32_t> dhead_peers{};
    KG_TRY(sym_alloc(c, (size_t)max_classes, &dkey, &dkey_peers));
    KG_TRY(sym_alloc(c, (size_t)max_classes, &dhead, &dhead_peers));
    if (n_classes)
        KG_LAUNCH(ctx, class_keys_kernel, grid_for(n_classes, kThreads, cap), kThreads, 0, sorted, head_pos.p, n_classes, g->core, g->deg, n,
                  key_mode, dkey, dhead);
    DevBuf<uint32_t> hist_total;
    DevBuf<double> lut, class_rank;
    KG_ALLOC(ctx, hist_total, n_bins);
    KG_ALLOC(ctx, lut, n_bins);
    KG_ALLOC(ctx, class_rank, n_classes);
    KG_LAUNCH(ctx, sum_peer_hist_kernel, grid_for(n_bins, kThreads, cap), kThreads, 0, hist_peers, world, n_bins, hist_total.p);
    KG_TRY((device_scan<uint32_t>(ctx, n_bins, HistIn{hist_total.p}, RankLutOut{lut.p, n}, (uint32_t *)nullptr)));
    unsigned long long token = 1, tokens[kMaxRanks];
    KG_TRY(comm_exchange(c, &token, 1, tokens));   // every rank's list is in place
    for (int q = 0; q < world; ++q) { L.key[q] = dkey_peers.p[q]; L.head[q] = dhead_peers.p[q]; }
    if (n_classes)
        KG_LAUNCH(ctx, class_rank_kernel, grid_for(n_classes, kThreads, cap), kThreads, 0, L, world, c->rank, n, class_rank.p);
    DevBuf<unsigned long long> max_bits(ctx, 1);
    if (!max_bits) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
    KG_CUDA(ctx, cudaMemsetAsync(max_bits.p, 0, sizeof(unsigned long long), ctx->stream));
    if (n_local)
        KG_LAUNCH(ctx, dist_score_kernel, grid_for(n_local, kThreads, cap), kThreads, 0, sorted, cls.p, class_rank.p, g->deg, lut.p, n_local,
                  g->score, max_bits.p);
    unsigned long long h_bits = 0, all_bits[kMaxRanks];
    KG_TRY(read_back(ctx, max_bits.p, &h_bits, 1));
    KG_TRY(comm_exchange(c, &h_bits, 1, all_bits));   // also: nobody releases lists a peer is still reading
    sym_release(c, mark);
    unsigned long long gmax = 0;
    for (int q = 0; q < world; ++q) gmax = all_bits[q] > gmax ? all_bits[q] : gmax;
    memcpy(&g->max_score, &gmax, sizeof(double));
    g->has_score = true;
    KG_CUDA(ctx, cudaEventRecord(ev1, ctx->stream));
    KG_CUDA(ctx, cudaEventSynchronize(ev1));
    cudaEventElapsedTime(&g->st.ms_corea, ev0, ev1);
    cudaEventDestroy(ev0);
    cudaEventDestroy(ev1);
    return KOMBGPU_OK;
}

}  // namespace kg
