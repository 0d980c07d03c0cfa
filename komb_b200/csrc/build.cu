// build.cu — stage 1 of the KOMB hot path on the device:
//   hits (read_key, unitig)  ->  per-read unitig sets  ->  clique pairs
//   ->  simple undirected edge set  ->  CSR of the symmetric graph.
//
// Restates, as sort/scan/compact kernels over integer arrays, what the reference
// does with string-keyed hash maps:
//   per-read set insert + mate union   src/graph.cpp:235,259-285   sort + adjacent-unique of (read, unitig)
//   all i<j pairs of every set         src/graph.cpp:332-347       segment scan + load-balanced pair emission
//   dedup / igraph_simplify            src/graph.cpp:342-347,438   sort + adjacent-unique of (min, max)
//   igraph_create adjacency index      src/graph.cpp:418           boundary detection + scan -> CSR
// No atomics are needed anywhere in this stage: every count falls out of run
// boundaries in sorted arrays, so the result (including the order inside each
// CSR row) is deterministic.
#include <cstdlib>

#include "graph.cuh"
#include "primitives.cuh"

namespace kg {

namespace {

constexpr int kThreads = 256;

inline uint32_t grid_for(uint64_t n, int per_block) { return ceil_div_u64(n ? n : 1, per_block); }

// ---- packing ---------------------------------------------------------------

// key = read_key << 32 | unitig; also the max read key (for the sort plan), an out-of-range flag, and how the
// read keys are ordered: info[0] = max read key, info[1] = error flag, info[2] = number of descents
// (read_key[i] < read_key[i-1]), info[3] = position of the first one.  SAM files list reads in input order, so the
// two mate files arrive as two runs of non-decreasing keys (one descent, at the file boundary).
__global__ void __launch_bounds__(kThreads) pack_hits_kernel(const uint32_t *__restrict__ read_key,
                                                             const uint32_t *__restrict__ unitig, uint64_t n_hits,
                                                             uint32_t n_vertices, uint64_t *__restrict__ keys,
                                                             uint32_t *__restrict__ info) {
    uint32_t local_max = 0, descents = 0, first = 0xffffffffu;
    bool bad = false;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_hits; i += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t r = read_key[i], u = unitig[i];
        bad |= (u >= n_vertices);
        local_max = max(local_max, r);
        if (i > 0 && r < read_key[i - 1]) { ++descents; first = min(first, (uint32_t)i); }
        keys[i] = ((uint64_t)r << 32) | u;
    }
    local_max = warp_reduce_max(local_max);
    descents = warp_reduce_add(descents);
    first = warp_reduce_min(first);
    if (lane_id() == 0) {
        if (local_max) atomicMax(&info[0], local_max);
        if (descents) { atomicAdd(&info[2], descents); atomicMin(&info[3], first); }
    }
    if (__any_sync(kFullMask, bad) && lane_id() == 0) atomicOr(&info[1], 1u);
}

// ---- reads in file order: merge the two runs, no sort -----------------------------------------------------

constexpr int kMergeItems = 8;
constexpr int kMergeTile = kThreads * kMergeItems;

__device__ __forceinline__ uint32_t read_of(uint64_t key) { return (uint32_t)(key >> 32); }

// number of A elements among the first `diag` outputs of the stable merge (A before B on equal read keys)
template <typename KeyA, typename KeyB>
__device__ __forceinline__ uint32_t merge_path(uint32_t diag, uint32_t n_a, uint32_t n_b, KeyA key_a, KeyB key_b) {
    uint32_t lo = diag > n_b ? diag - n_b : 0, hi = min(diag, n_a);
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (key_a(mid) <= key_b(diag - 1 - mid)) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// part[t] = A elements before output t * kMergeTile
__global__ void __launch_bounds__(kThreads) merge_partition_kernel(const uint64_t *__restrict__ a, uint32_t n_a,
                                                                   const uint64_t *__restrict__ b, uint32_t n_b,
                                                                   uint32_t n_tiles, uint32_t *__restrict__ part) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t > n_tiles) return;
    const uint32_t diag = (uint32_t)min((uint64_t)t * kMergeTile, (uint64_t)n_a + n_b);
    part[t] = merge_path(diag, n_a, n_b, [&](uint32_t i) { return read_of(a[i]); }, [&](uint32_t j) { return read_of(b[j]); });
}

// stable merge by read key of two runs of packed hits; the unitigs of a read stay in arrival order
__global__ void __launch_bounds__(kThreads) merge_runs_kernel(const uint64_t *__restrict__ a, uint32_t n_a,
                                                              const uint64_t *__restrict__ b, uint32_t n_b,
                                                              const uint32_t *__restrict__ part, uint64_t *__restrict__ out) {
    __shared__ uint64_t s_key[kMergeTile];
    const uint32_t tile = blockIdx.x;
    const uint64_t o0 = (uint64_t)tile * kMergeTile;
    const uint32_t count = (uint32_t)min((uint64_t)kMergeTile, (uint64_t)n_a + n_b - o0);
    const uint32_t a0 = part[tile], a1 = part[tile + 1];
    const uint32_t b0 = (uint32_t)(o0 - a0);
    const uint32_t ca = a1 - a0, cb = count - ca;   // the tile's A keys sit at s_key[0, ca), its B keys behind them
    for (uint32_t i = threadIdx.x; i < count; i += kThreads) s_key[i] = i < ca ? a[a0 + i] : b[b0 + (i - ca)];
    __syncthreads();
    const uint32_t diag = min(threadIdx.x * kMergeItems, count);
    uint32_t ia = merge_path(diag, ca, cb, [&](uint32_t i) { return read_of(s_key[i]); },
                             [&](uint32_t j) { return read_of(s_key[ca + j]); });
    uint32_t ib = diag - ia;
    uint64_t res[kMergeItems];
#pragma unroll
    for (int j = 0; j < kMergeItems; ++j) {
        const bool has_a = ia < ca, has_b = ib < cb;
        const uint64_t ka = has_a ? s_key[ia] : 0, kb = has_b ? s_key[ca + ib] : 0;
        const bool take_a = has_a && (!has_b || read_of(ka) <= read_of(kb));
        res[j] = take_a ? ka : kb;
        if (take_a) ++ia; else ++ib;
    }
#pragma unroll
    for (int j = 0; j < kMergeItems; ++j)
        if (diag + j < count) out[o0 + diag + j] = res[j];
}

// hits grouped by read (unitigs in any order inside a read): 1 for the first occurrence of a (read, unitig).
// A read longer than kMaxReadScan hits is left to the general sort path (*too_long is raised).
constexpr uint32_t kMaxReadScan = 64;
struct FirstInReadFlag {
    const uint64_t *hits;
    uint32_t *too_long;
    __device__ uint32_t operator()(uint64_t i) const {
        const uint64_t k = hits[i];
        for (uint32_t back = 1; back <= i; ++back) {
            const uint64_t p = hits[i - back];
            if ((p >> 32) != (k >> 32)) return 1u;
            if (p == k) return 0u;
            if (back == kMaxReadScan) { atomicExch(too_long, 1u); return 1u; }
        }
        return 1u;
    }
};

// canonical undirected key (min << 32 | max); loops keep u == v and are dropped
// by the unique pass.
__global__ void __launch_bounds__(kThreads) pack_pairs_kernel(const uint32_t *__restrict__ u, const uint32_t *__restrict__ v,
                                                              uint64_t n_pairs, uint32_t n_vertices,
                                                              uint64_t *__restrict__ keys, uint32_t *__restrict__ info) {
    bool bad = false;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_pairs; i += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t a = u[i], b = v[i];
        bad |= (a >= n_vertices) | (b >= n_vertices);
        uint32_t lo = min(a, b), hi = max(a, b);
        keys[i] = ((uint64_t)lo << 32) | hi;
    }
    if (__any_sync(kFullMask, bad) && lane_id() == 0) atomicOr(&info[1], 1u);
}

// ---- per-read segments -------------------------------------------------------

// A "good" segment is a read with >= 2 distinct unitigs.  hi word counts good
// heads, lo word counts good tails; the s-th good head and the s-th good tail
// delimit the s-th good segment.
struct SegFlagIn {
    const uint64_t *hits;  // sorted unique (read << 32 | unitig)
    uint64_t n;
    __device__ uint64_t operator()(uint64_t i) const {
        uint32_t r = (uint32_t)(hits[i] >> 32);
        bool same_prev = i > 0 && (uint32_t)(hits[i - 1] >> 32) == r;
        bool same_next = i + 1 < n && (uint32_t)(hits[i + 1] >> 32) == r;
        uint64_t head = (!same_prev && same_next) ? 1ull : 0ull;
        uint64_t tail = (same_prev && !same_next) ? 1ull : 0ull;
        return (head << 32) | tail;
    }
};
struct SegFlagOut {
    uint32_t *seg_head;
    uint32_t *seg_tail;
    __device__ void operator()(uint64_t i, uint64_t prefix, uint64_t v) const {
        if (v >> 32) seg_head[prefix >> 32] = (uint32_t)i;
        if (v & 0xffffffffu) seg_tail[prefix & 0xffffffffu] = (uint32_t)i;
    }
};

// pairs of segment s = C(size, 2)
struct SegPairsIn {
    const uint32_t *seg_head;
    const uint32_t *seg_tail;
    __device__ uint64_t operator()(uint64_t s) const {
        uint64_t k = (uint64_t)(seg_tail[s] - seg_head[s]) + 1;
        return k * (k - 1) / 2;
    }
};
struct SegPairsOut {
    uint64_t *seg_base;
    __device__ void operator()(uint64_t s, uint64_t prefix, uint64_t) const { seg_base[s] = prefix; }
};

// ---- load-balanced pair emission ----------------------------------------------

constexpr int kEmitItems = 8;
constexpr int kEmitTile = kThreads * kEmitItems;  // outputs per CTA

// Pairs [base, end) of the global pair index are emitted to pairs[0, end - base): the whole list in one shot (base 0)
// or one chunk of it.  tile_seg[t] = last segment s with seg_base[s] <= base + t * kEmitTile
__global__ void __launch_bounds__(kThreads) emit_partition_kernel(const uint64_t *__restrict__ seg_base, uint32_t n_seg,
                                                                  uint32_t n_tiles, uint64_t base, uint32_t *__restrict__ tile_seg) {
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_tiles) return;
    uint64_t p = base + (uint64_t)t * kEmitTile;
    uint32_t lo = 0, hi = n_seg;  // invariant: seg_base[lo] <= p, (hi == n_seg or seg_base[hi] > p)
    while (hi - lo > 1) {
        uint32_t mid = lo + (hi - lo) / 2;
        if (seg_base[mid] <= p) lo = mid; else hi = mid;
    }
    tile_seg[t] = lo;
}

__global__ void __launch_bounds__(kThreads) emit_pairs_kernel(const uint64_t *__restrict__ hits,
                                                              const uint32_t *__restrict__ seg_head,
                                                              const uint64_t *__restrict__ seg_base, uint32_t n_seg,
                                                              const uint32_t *__restrict__ tile_seg, uint32_t n_tiles,
                                                              uint64_t base, uint64_t end, uint64_t *__restrict__ pairs) {
    __shared__ uint64_t s_base[kEmitTile + 2];
    __shared__ uint32_t s_head[kEmitTile + 2];
    const uint32_t tile = blockIdx.x;
    const uint64_t p0 = base + (uint64_t)tile * kEmitTile;
    const uint64_t p1 = min(end, p0 + kEmitTile);
    const uint32_t s_first = tile_seg[tile];
    const uint32_t s_last = tile + 1 < n_tiles ? tile_seg[tile + 1] : n_seg - 1;
    // every segment is non-empty, so the tile's pairs lie in its first kEmitTile segments (the last tile of a chunk
    // may see every later segment up to n_seg - 1)
    const uint32_t cnt = min(s_last - s_first + 1, (uint32_t)kEmitTile + 1);
    for (uint32_t i = threadIdx.x; i < cnt; i += kThreads) {
        s_base[i] = seg_base[s_first + i];
        s_head[i] = seg_head[s_first + i];
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < kEmitItems; ++j) {
        uint64_t p = p0 + (uint64_t)j * kThreads + threadIdx.x;
        if (p >= p1) break;
        uint32_t lo = 0, hi = cnt;
        while (hi - lo > 1) {
            uint32_t mid = (lo + hi) >> 1;
            if (s_base[mid] <= p) lo = mid; else hi = mid;
        }
        // t-th pair (a < b) of the segment in colexicographic order: t = b(b-1)/2 + a
        uint64_t t = p - s_base[lo];
        uint64_t b = (uint64_t)((1.0 + sqrt(1.0 + 8.0 * (double)t)) * 0.5);
        while (b * (b - 1) / 2 > t) --b;
        while ((b + 1) * b / 2 <= t) ++b;
        uint64_t a = t - b * (b - 1) / 2;
        const uint64_t h = s_head[lo];
        const uint32_t ua = (uint32_t)hits[h + a], ub = (uint32_t)hits[h + b];  // distinct; ascending only after a sort
        pairs[p - base] = ((uint64_t)min(ua, ub) << 32) | max(ua, ub);
    }
}

// ---- unique of sorted pair keys, dropping loops ---------------------------------

struct EdgeFlagIn {
    const uint64_t *keys;
    __device__ uint32_t operator()(uint64_t i) const {
        uint64_t k = keys[i];
        bool head = (i == 0 || keys[i - 1] != k);
        bool loop = (uint32_t)(k >> 32) == (uint32_t)k;
        return (head && !loop) ? 1u : 0u;
    }
};

// adjacent-unique of the sorted pair keys that also records how many pairs collapsed into each edge (the number of
// reads supporting it: the "weight" of the north star's weighted graph; the reference itself keeps no weights,
// src/graph.cpp:438 passes comb = NULL).  Runs are short (1.0005 pairs per edge on cfg2), so the head looks ahead a
// few keys and only then falls back to a binary search for the end of its run.
struct CompactEdgesMult {
    const uint64_t *keys;
    uint64_t n;
    uint64_t *dst;
    uint32_t *mult;
    __device__ void operator()(uint64_t i, uint32_t pos, uint32_t flag) const {
        if (!flag) return;
        const uint64_t k = keys[i];
        dst[pos] = k;
        uint64_t r = 1;
        while (r < 8 && i + r < n && keys[i + r] == k) ++r;
        if (r == 8 && i + r < n && keys[i + r] == k) {
            uint64_t lo = i + r, hi = n;   // first position past i + r whose key differs
            while (lo < hi) {
                const uint64_t mid = lo + (hi - lo) / 2;
                if (keys[mid] == k) lo = mid + 1; else hi = mid;
            }
            r = lo - i;
        }
        mult[pos] = (uint32_t)r;
    }
};

// ---- chunked path: merge of two sorted unique (key, count) lists ---------------------------------------------
// A is the running edge list, B one chunk's.  Merge path over the merged sequence with both copies of a shared key
// (A's first); a B key equal to the A key before it is a duplicate: it is dropped and its count added to A's.  An
// output lands at its merged position minus the duplicates before it, so one counting pass (duplicates per tile)
// and a scan over the tiles give every write position, and the output size is known before it is allocated.

// part[t] = A elements among the first t * kMergeTile merged elements (A before B on equal keys)
__global__ void __launch_bounds__(kThreads) unique_merge_partition_kernel(const uint64_t *__restrict__ a, uint64_t n_a,
                                                                          const uint64_t *__restrict__ b, uint64_t n_b,
                                                                          uint32_t n_tiles, uint64_t *__restrict__ part) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t > n_tiles) return;
    const uint64_t diag = min((uint64_t)t * kMergeTile, n_a + n_b);
    uint64_t lo = diag > n_b ? diag - n_b : 0, hi = min(diag, n_a);
    while (lo < hi) {
        const uint64_t mid = lo + (hi - lo) / 2;
        if (a[mid] <= b[diag - 1 - mid]) lo = mid + 1; else hi = mid;
    }
    part[t] = lo;
}

// kWrite = false: tile_dups[t] = B duplicates in tile t.  kWrite = true: tile_dups[t] = duplicates in the tiles before
// t; writes the merged unique keys and their summed counts (saturating at 2^32 - 1).
template <bool kWrite>
__global__ void __launch_bounds__(kThreads) unique_merge_kernel(const uint64_t *__restrict__ a, const uint32_t *__restrict__ a_cnt,
                                                                uint64_t n_a, const uint64_t *__restrict__ b,
                                                                const uint32_t *__restrict__ b_cnt, uint64_t n_b,
                                                                const uint64_t *__restrict__ part, uint32_t *__restrict__ tile_dups,
                                                                uint64_t *__restrict__ out, uint32_t *__restrict__ out_cnt) {
    // s_key = [A[a0 - 1] | the tile's A keys | its B keys | B[b0 + cb]]; ~0 (a loop, never a key) where absent
    __shared__ uint64_t s_key[kMergeTile + 2];
    __shared__ uint32_t s_scan[kThreads / 32 + 1];
    const uint32_t tile = blockIdx.x;
    const uint64_t o0 = (uint64_t)tile * kMergeTile;
    const uint32_t count = (uint32_t)min((uint64_t)kMergeTile, n_a + n_b - o0);
    const uint64_t a0 = part[tile], b0 = o0 - a0;
    const uint32_t ca = (uint32_t)(part[tile + 1] - a0), cb = count - ca;
    for (uint32_t i = threadIdx.x; i < count + 2; i += kThreads) {
        uint64_t k = ~0ull;
        if (i == 0) { if (a0 > 0) k = a[a0 - 1]; }
        else if (i <= ca) k = a[a0 + i - 1];
        else if (i <= count) k = b[b0 + (i - 1 - ca)];
        else if (b0 + cb < n_b) k = b[b0 + cb];
        s_key[i] = k;
    }
    __syncthreads();
    const uint64_t *s_a = s_key + 1, *s_b = s_key + 1 + ca;   // s_a[-1] = A[a0 - 1], s_b[cb] = B[b0 + cb]
    const uint32_t diag = min(threadIdx.x * kMergeItems, count);
    const uint32_t ia0 = merge_path(diag, ca, cb, [&](uint32_t i) { return s_a[i]; }, [&](uint32_t j) { return s_b[j]; });
    const uint32_t ib0 = diag - ia0;
    uint32_t ia = ia0, ib = ib0, dups = 0;
#pragma unroll
    for (int j = 0; j < kMergeItems; ++j) {
        if (diag + j >= count) break;
        if (ia < ca && (ib >= cb || s_a[ia] <= s_b[ib])) ++ia;
        else { dups += s_a[(int)ia - 1] == s_b[ib]; ++ib; }
    }
    uint32_t tile_total;
    const uint32_t before = block_excl_scan_add<uint32_t, kThreads>(dups, s_scan, &tile_total);
    if (!kWrite) {
        if (threadIdx.x == 0) tile_dups[tile] = tile_total;
        return;
    }
    uint64_t pos = o0 + diag - tile_dups[tile] - before;
    ia = ia0; ib = ib0;
#pragma unroll
    for (int j = 0; j < kMergeItems; ++j) {
        if (diag + j >= count) break;
        if (ia < ca && (ib >= cb || s_a[ia] <= s_b[ib])) {
            const uint64_t k = s_a[ia];
            uint64_t c = a_cnt[a0 + ia];
            if (s_b[ib] == k) c += b_cnt[b0 + ib];   // its B copy follows (possibly in the next tile)
            out[pos] = k;
            out_cnt[pos] = (uint32_t)min(c, (uint64_t)0xffffffffu);
            ++pos; ++ia;
        } else {
            const uint64_t k = s_b[ib];
            if (s_a[(int)ia - 1] != k) { out[pos] = k; out_cnt[pos] = b_cnt[b0 + ib]; ++pos; }
            ++ib;
        }
    }
}

struct ReadU32 {
    const uint32_t *x;
    __device__ uint32_t operator()(uint64_t i) const { return x[i]; }
};
struct WriteU32Prefix {
    uint32_t *x;
    __device__ void operator()(uint64_t i, uint32_t prefix, uint32_t) const { x[i] = prefix; }
};

// ---- CSR ---------------------------------------------------------------------------

__global__ void __launch_bounds__(kThreads) swap_pack_kernel(const uint64_t *__restrict__ edges, uint64_t n_edges,
                                                             uint64_t *__restrict__ swapped) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_edges; i += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t e = edges[i];
        swapped[i] = (e << 32) | (e >> 32);
    }
}

// keys sorted by their high word, which lies in [base, base + n_rows): start[x] = first index whose high word is
// >= base + x, for x in [0, n_rows]  (start[n_rows] = count).  No atomics on the result: thread i fills the rows between
// its predecessor's and its own -- but only short gaps; a long run of empty rows (a rank of the partitioned path sees
// only the neighbourhood of its own id range; an edge list may leave whole id ranges without edges) is recorded and
// filled by a whole CTA in a second kernel, so one thread never writes millions of entries.
// *err (optional) is raised when a key lies outside [base, base + n_rows) or its low word is >= lo_bound.
constexpr int64_t kGapShort = 32;
struct RowGap {
    uint32_t lo, hi, val;   // start[lo .. hi] = val
};
__global__ void __launch_bounds__(kThreads) row_bounds_kernel(const uint64_t *__restrict__ keys, uint64_t count, uint32_t base,
                                                              uint32_t n_rows, uint32_t lo_bound, uint32_t *__restrict__ start,
                                                              RowGap *__restrict__ gaps, uint32_t *__restrict__ n_gaps, uint32_t *__restrict__ err) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i <= count; i += (uint64_t)gridDim.x * blockDim.x) {
        int64_t cur = (int64_t)n_rows, prev = -1;
        if (i < count) {
            const uint64_t k = keys[i];
            cur = (int64_t)(uint32_t)(k >> 32) - (int64_t)base;
            if (cur < 0 || cur >= (int64_t)n_rows || (uint32_t)k >= lo_bound) {
                if (err) atomicExch(err, 2u);
                cur = (int64_t)n_rows;
            }
        }
        if (i > 0) {
            prev = (int64_t)(uint32_t)(keys[i - 1] >> 32) - (int64_t)base;
            if (prev < 0 || prev >= (int64_t)n_rows) prev = (int64_t)n_rows;
        }
        if (cur - prev > kGapShort) {
            const uint32_t g = atomicAdd(n_gaps, 1u);
            gaps[g] = RowGap{(uint32_t)(prev + 1), (uint32_t)cur, (uint32_t)i};
        } else {
            for (int64_t x = prev + 1; x <= cur; ++x) start[x] = (uint32_t)i;
        }
    }
}
__global__ void __launch_bounds__(kThreads) row_gaps_kernel(const RowGap *__restrict__ gaps, const uint32_t *__restrict__ n_gaps,
                                                            uint32_t *__restrict__ start) {
    const uint32_t n = *n_gaps;
    for (uint32_t g = blockIdx.x; g < n; g += gridDim.x) {
        const RowGap gp = gaps[g];
        for (uint64_t x = (uint64_t)gp.lo + threadIdx.x; x <= gp.hi; x += blockDim.x) start[x] = gp.val;
    }
}

struct DegreeIn {
    const uint32_t *fwd_start;
    const uint32_t *back_start;
    __device__ uint64_t operator()(uint64_t v) const {
        return (uint64_t)(fwd_start[v + 1] - fwd_start[v]) + (uint64_t)(back_start[v + 1] - back_start[v]);
    }
};
struct DegreeOut {
    uint64_t *row_ptr;
    int32_t *deg;
    __device__ void operator()(uint64_t v, uint64_t prefix, uint64_t d) const {
        row_ptr[v] = prefix;
        deg[v] = (int32_t)d;
    }
};

// max of an int32 array: warp shuffle -> one atomic per warp
__global__ void __launch_bounds__(kThreads) reduce_max_i32_kernel(const int32_t *__restrict__ x, uint64_t n,
                                                                  int32_t *__restrict__ out) {
    int32_t m = INT32_MIN;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
        m = max(m, x[i]);
    m = warp_reduce_max(m);
    if (lane_id() == 0 && m != INT32_MIN) atomicMax(out, m);
}

// Row v = [back neighbours (< v, ascending) | forward neighbours (> v, ascending)].
__global__ void __launch_bounds__(kThreads) fill_col_kernel(const uint64_t *__restrict__ edges,
                                                            const uint64_t *__restrict__ swapped, uint64_t n_edges,
                                                            const uint64_t *__restrict__ row_ptr,
                                                            const uint32_t *__restrict__ fwd_start,
                                                            const uint32_t *__restrict__ back_start,
                                                            uint32_t *__restrict__ col) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_edges; i += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t e = edges[i];
        uint32_t u = (uint32_t)(e >> 32);
        uint64_t nback = back_start[u + 1] - back_start[u];
        col[row_ptr[u] + nback + (i - fwd_start[u])] = (uint32_t)e;
        uint64_t s = swapped[i];
        uint32_t v = (uint32_t)(s >> 32);
        col[row_ptr[v] + (i - back_start[v])] = (uint32_t)s;
    }
}

__global__ void set_u64_kernel(uint64_t *p, uint64_t v) { *p = v; }

// keys sorted by high word: idx[j] = first position whose high word is >= bounds[j]
__global__ void lower_bounds_kernel(const uint64_t *__restrict__ keys, uint64_t count, const uint32_t *__restrict__ bounds,
                                    int nb, uint64_t *__restrict__ idx) {
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nb) return;
    const uint64_t target = (uint64_t)bounds[j] << 32;
    uint64_t lo = 0, hi = count;  // first position with keys[pos] >= target
    while (lo < hi) {
        uint64_t mid = lo + (hi - lo) / 2;
        if (keys[mid] < target) lo = mid + 1; else hi = mid;
    }
    idx[j] = lo;
}

// row r of a partition owns the keys whose high word is base + r
// *err is raised when a key's row lies outside [base, base + n_rows) or its low word is >= lo_bound (an entry routed to
// the wrong rank, or a corrupt one, must not write past the arrays)
__global__ void __launch_bounds__(kThreads) row_bounds_base_kernel(const uint64_t *__restrict__ keys, uint64_t count,
                                                                   uint32_t base, uint32_t n_rows, uint32_t lo_bound,
                                                                   uint64_t *__restrict__ start, uint32_t *__restrict__ err) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i <= count; i += (uint64_t)gridDim.x * blockDim.x) {
        int64_t cur = (int64_t)n_rows, prev = -1;
        if (i < count) {
            const uint64_t k = keys[i];
            cur = (int64_t)(uint32_t)(k >> 32) - (int64_t)base;
            if (cur < 0 || cur >= (int64_t)n_rows || (uint32_t)k >= lo_bound) { atomicExch(err, 2u); cur = (int64_t)n_rows; }
        }
        if (i > 0) {
            prev = (int64_t)(uint32_t)(keys[i - 1] >> 32) - (int64_t)base;
            if (prev < 0 || prev >= (int64_t)n_rows) prev = (int64_t)n_rows;
        }
        for (int64_t x = prev + 1; x <= cur; ++x) start[x] = i;
    }
}

__global__ void __launch_bounds__(kThreads) part_cols_kernel(const uint64_t *__restrict__ keys, uint64_t count,
                                                             uint32_t *__restrict__ col) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (uint64_t)gridDim.x * blockDim.x)
        col[i] = (uint32_t)keys[i];
}

__global__ void __launch_bounds__(kThreads) part_degree_kernel(const uint64_t *__restrict__ row_ptr, uint32_t n_rows,
                                                               int32_t *__restrict__ deg, int32_t *__restrict__ max_deg) {
    int32_t m = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_rows; i += (uint64_t)gridDim.x * blockDim.x) {
        int32_t d = (int32_t)(row_ptr[i + 1] - row_ptr[i]);
        deg[i] = d;
        m = max(m, d);
    }
    m = warp_reduce_max(m);
    if (lane_id() == 0 && m) atomicMax(max_deg, m);
}

struct AnyHeadFlag {  // unique of sorted directed entries (no loop test: routed entries never hold loops)
    const uint64_t *keys;
    __device__ uint32_t operator()(uint64_t i) const { return (i == 0 || keys[i] != keys[i - 1]) ? 1u : 0u; }
};

// ---- chunked path -----------------------------------------------------------------------------------------------
// A clique of k unitigs emits C(k, 2) pairs, so P outgrows the edge count E by far on repeats.  When P reaches 2^32 (or
// exceeds KOMBGPU_PAIR_CHUNK), the pairs are emitted, sorted and reduced to (key, count) a chunk at a time, and each
// chunk is merged into the running edge list: device memory holds one chunk of pairs plus O(E + H).

// the chunk size when P takes the chunked path, else 0
uint64_t pair_chunk(uint64_t n_pairs) {
    const uint64_t cap = pair_chunk_env();
    if (cap && n_pairs > cap) return min(cap, (uint64_t)0xffffffffu);   // a chunk's counts are 32-bit
    return n_pairs >= (1ull << 32) ? kPairChunk : 0;
}

// where the edge list (and its multiplicities) go when the chunked path runs
struct EdgeSink {
    DevBuf<uint64_t> *edges;
    uint64_t *n_edges;
    DevBuf<uint32_t> *mult;   // optional
    uint32_t *n_chunks;       // optional
};

// emit(p0, p1, dst) writes the canonical keys of pairs [p0, p1) to dst[0, p1 - p0)
template <typename Emit>
int chunked_edges(kombgpu_ctx *ctx, uint64_t n_pairs, uint64_t chunk, int bn, Emit emit, EdgeSink *sink) {
    DevBuf<uint64_t> ka, kb;
    DevBuf<uint32_t> ccnt;
    KG_ALLOC(ctx, ka, chunk);
    KG_ALLOC(ctx, kb, chunk);
    KG_ALLOC(ctx, ccnt, chunk);
    RadixPass passes[8];
    const int np = plan_radix_passes(0, bn, 32, 32 + bn, passes);
    EdgeRun run;
    uint32_t n_chunks = 0;
    for (uint64_t p0 = 0; p0 < n_pairs; p0 += chunk, ++n_chunks) {
        const uint64_t n_c = min(chunk, n_pairs - p0);
        // emit, sort, reduce to sorted unique (key, count) in the other ping-pong buffer, merge into the running list
        KG_TRY(emit(p0, p0 + n_c, ka.p));
        uint64_t *sorted = ka.p;
        KG_TRY(radix_sort_u64(ctx, ka.p, kb.p, n_c, passes, np, &sorted));
        KG_TRY(merge_sorted_chunk(ctx, sorted, n_c, sorted == ka.p ? kb.p : ka.p, ccnt.p, &run));
    }
    if (!run.keys) KG_ALLOC(ctx, run.keys, 0);
    *sink->edges = std::move(run.keys);
    *sink->n_edges = run.n;
    if (sink->mult) {
        if (!run.cnt) KG_ALLOC(ctx, run.cnt, 0);
        *sink->mult = std::move(run.cnt);
    }
    if (sink->n_chunks) *sink->n_chunks = n_chunks;
    return KOMBGPU_OK;
}

// (u, v) pairs -> canonical keys, sorted (duplicates and loops still in)
int pairs_to_sorted_keys(kombgpu_ctx *ctx, const uint32_t *u, const uint32_t *v, uint64_t n_pairs, uint32_t n_vertices,
                         DevBuf<uint64_t> &ka, DevBuf<uint64_t> &kb, uint64_t **sorted_out) {
    if (n_pairs >= (1ull << 32)) return ctx_fail(ctx, KOMBGPU_EINVAL, "n_pairs >= 2^32 is not supported on one device");
    const int bn = bits_for(n_vertices > 0 ? n_vertices - 1 : 0);
    DevBuf<uint32_t> info(ctx, 2);
    KG_ALLOC(ctx, ka, n_pairs);
    KG_ALLOC(ctx, kb, n_pairs);
    if (!info) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
    KG_CUDA(ctx, cudaMemsetAsync(info.p, 0, 2 * sizeof(uint32_t), ctx->stream));
    uint64_t *sorted = ka.p;
    if (n_pairs) {
        KG_LAUNCH(ctx, pack_pairs_kernel, min(grid_for(n_pairs, kThreads), 148u * 16u), kThreads, 0, u, v, n_pairs, n_vertices,
                  ka.p, info.p);
        RadixPass passes[8];
        int np = plan_radix_passes(0, bn, 32, 32 + bn, passes);
        KG_TRY(radix_sort_u64(ctx, ka.p, kb.p, n_pairs, passes, np, &sorted));
    }
    uint32_t h_info[2] = {0, 0};
    KG_TRY(read_back(ctx, info.p, h_info, 2));
    if (h_info[1]) return ctx_fail(ctx, KOMBGPU_EINVAL, "edge endpoint >= n_vertices (%u)", n_vertices);
    *sorted_out = sorted;
    return KOMBGPU_OK;
}

}  // namespace

// sorted pair keys (duplicates, loops possible) -> unique simple edges
int unique_edges(kombgpu_ctx *ctx, const uint64_t *keys, uint64_t count, DevBuf<uint64_t> &edges, uint64_t *n_edges,
                 DevBuf<uint32_t> *mult) {
    DevBuf<uint32_t> d_count(ctx, 1);
    if (!d_count) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
    KG_ALLOC(ctx, edges, count);
    if (mult) {
        KG_ALLOC(ctx, *mult, count);
        KG_TRY((device_scan<uint32_t>(ctx, count, EdgeFlagIn{keys}, CompactEdgesMult{keys, count, edges.p, mult->p}, d_count.p)));
    } else
    KG_TRY((device_scan<uint32_t>(ctx, count, EdgeFlagIn{keys}, CompactKeysU64{keys, edges.p}, d_count.p)));
    uint32_t n32 = 0;
    KG_TRY(read_back(ctx, d_count.p, &n32, 1));
    *n_edges = n32;
    return KOMBGPU_OK;
}

// (v << 32 | u) copy of an edge list, stably sorted on v: the backward half of the adjacency in order
int swapped_sorted(kombgpu_ctx *ctx, const uint64_t *edges, uint64_t n_edges, uint32_t n_vertices, DevBuf<uint64_t> &a,
                   DevBuf<uint64_t> &b, uint64_t **out) {
    const int bn = bits_for(n_vertices > 0 ? n_vertices - 1 : 0);
    KG_ALLOC(ctx, a, n_edges);
    KG_ALLOC(ctx, b, n_edges);
    *out = a.p;
    if (n_edges) {
        KG_LAUNCH(ctx, swap_pack_kernel, min(grid_for(n_edges, kThreads), 148u * 16u), kThreads, 0, edges, n_edges, a.p);
        RadixPass passes[8];
        int np = plan_radix_passes(32, 32 + bn, 0, 0, passes);
        KG_TRY(radix_sort_u64(ctx, a.p, b.p, n_edges, passes, np, out));
    }
    return KOMBGPU_OK;
}

int lower_bounds_hi(kombgpu_ctx *ctx, const uint64_t *keys, uint64_t count, const uint32_t *bounds_host, int nb,
                    uint64_t *idx_host) {
    DevBuf<uint32_t> d_b;
    DevBuf<uint64_t> d_i;
    KG_ALLOC(ctx, d_b, nb);
    KG_ALLOC(ctx, d_i, nb);
    KG_CUDA(ctx, cudaMemcpyAsync(d_b.p, bounds_host, nb * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    KG_LAUNCH(ctx, lower_bounds_kernel, 1, 64, 0, keys, count, d_b.p, nb, d_i.p);
    return read_back(ctx, d_i.p, idx_host, nb);
}

uint64_t pair_chunk_env() {
    const char *e = getenv("KOMBGPU_PAIR_CHUNK");   // tests and A/B runs
    return e ? strtoull(e, nullptr, 10) : 0;
}

int merge_sorted_chunk(kombgpu_ctx *ctx, const uint64_t *sorted, uint64_t n_c, uint64_t *cuniq, uint32_t *ccnt, EdgeRun *run) {
    DevBuf<uint32_t> d_cnt(ctx, 1);
    if (!d_cnt) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
    KG_TRY((device_scan<uint32_t>(ctx, n_c, EdgeFlagIn{sorted}, CompactEdgesMult{sorted, n_c, cuniq, ccnt}, d_cnt.p)));
    uint32_t n_u = 0;
    KG_TRY(read_back(ctx, d_cnt.p, &n_u, 1));
    if (n_u == 0) return KOMBGPU_OK;
    // merge into the running list: count the duplicates per tile, then the output size, then write
    const uint64_t n_run = run->n, n_m = n_run + n_u;
    const uint32_t n_tiles = ceil_div_u64(n_m, kMergeTile);
    DevBuf<uint64_t> part, next;
    DevBuf<uint32_t> tile_dups, next_cnt;
    KG_ALLOC(ctx, part, (size_t)n_tiles + 1);
    KG_ALLOC(ctx, tile_dups, n_tiles);
    KG_LAUNCH(ctx, unique_merge_partition_kernel, grid_for((uint64_t)n_tiles + 1, kThreads), kThreads, 0, run->keys.p, n_run, cuniq,
              (uint64_t)n_u, n_tiles, part.p);
    KG_LAUNCH(ctx, unique_merge_kernel<false>, n_tiles, kThreads, 0, run->keys.p, run->cnt.p, n_run, cuniq, ccnt, (uint64_t)n_u,
              part.p, tile_dups.p, nullptr, nullptr);
    KG_TRY((device_scan<uint32_t>(ctx, n_tiles, ReadU32{tile_dups.p}, WriteU32Prefix{tile_dups.p}, d_cnt.p)));
    uint32_t n_dups = 0;
    KG_TRY(read_back(ctx, d_cnt.p, &n_dups, 1));
    const uint64_t n_out = n_m - n_dups;
    if (n_out >= (1ull << 32))
        return ctx_fail(ctx, KOMBGPU_EINVAL, "%llu simple edges exceed the 2^32 per-device edge limit", (unsigned long long)n_out);
    KG_ALLOC(ctx, next, n_out);
    KG_ALLOC(ctx, next_cnt, n_out);
    KG_LAUNCH(ctx, unique_merge_kernel<true>, n_tiles, kThreads, 0, run->keys.p, run->cnt.p, n_run, cuniq, ccnt, (uint64_t)n_u,
              part.p, tile_dups.p, next.p, next_cnt.p);
    // the running list only grows: give the old one back to the device rather than to the context's cache
    ws_release(ctx, run->keys.take());
    ws_release(ctx, run->cnt.take());
    run->keys = std::move(next);
    run->cnt = std::move(next_cnt);
    run->n = n_out;
    return KOMBGPU_OK;
}

int HitPairs::emit(uint64_t p0, uint64_t p1, uint64_t *dst) {
    if (p1 <= p0) return KOMBGPU_OK;
    const uint32_t n_tiles = ceil_div_u64(p1 - p0, kEmitTile);
    if (tile_seg.count < n_tiles) KG_ALLOC(ctx, tile_seg, n_tiles);
    KG_LAUNCH(ctx, emit_partition_kernel, grid_for(n_tiles, kThreads), kThreads, 0, seg_base.p, n_seg, n_tiles, p0, tile_seg.p);
    KG_LAUNCH(ctx, emit_pairs_kernel, n_tiles, kThreads, 0, hits, seg_head.p, seg_base.p, n_seg, tile_seg.p, n_tiles, p0, p1, dst);
    return KOMBGPU_OK;
}

void HitPairs::release() {
    ha.release(); hb.release(); hc.release(); seg_base.release();
    seg_head.release(); seg_tail.release(); tile_seg.release();
    hits = nullptr;
}

int count_hit_pairs(kombgpu_ctx *ctx, const uint32_t *read_key, const uint32_t *unitig, uint64_t n_hits, uint32_t n_vertices,
                    HitPairs *hp, kombgpu_stats *st) {
    if (n_hits >= (1ull << 32)) return ctx_fail(ctx, KOMBGPU_EINVAL, "n_hits >= 2^32 is not supported on one device");
    const int bn = bits_for(n_vertices > 0 ? n_vertices - 1 : 0);
    hp->ctx = ctx;
    st->n_hits = n_hits;
    DevBuf<uint64_t> &ha = hp->ha, &hb = hp->hb;

    // 1. (read, unitig) keys, sorted + unique  == per-read unitig SETS, mates merged
    DevBuf<uint32_t> info(ctx, 5);
    KG_ALLOC(ctx, ha, n_hits);
    KG_ALLOC(ctx, hb, n_hits);
    if (!info) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
    const uint32_t info0[5] = {0, 0, 0, 0xffffffffu, 0};   // max key, error, descents, first descent, read too long
    KG_CUDA(ctx, cudaMemcpyAsync(info.p, info0, sizeof(info0), cudaMemcpyHostToDevice, ctx->stream));
    if (n_hits)
        KG_LAUNCH(ctx, pack_hits_kernel, min(grid_for(n_hits, kThreads), 148u * 16u), kThreads, 0, read_key, unitig, n_hits,
                  n_vertices, ha.p, info.p);
    uint32_t h_info[5] = {0, 0, 0, 0, 0};
    KG_TRY(read_back(ctx, info.p, h_info, 5));
    if (h_info[1]) return ctx_fail(ctx, KOMBGPU_EINVAL, "unitig id >= n_vertices (%u)", n_vertices);
    DevBuf<uint32_t> d_cnt(ctx, 1);
    if (!d_cnt) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
    uint64_t *sorted = ha.p, *other = hb.p;
    uint32_t n_uniq = 0;
    RadixPass passes[8];
    bool grouped = false;   // unique hits grouped by read without a sort?
    if (n_hits && h_info[2] <= 1 && !getenv("KOMBGPU_NO_MERGE")) {
        // The reads arrive in file order (at most two runs of non-decreasing keys: the two mate files): a stable
        // merge by read key replaces the radix sort (6 passes for cfg2), and since the per-read unitig SET is all
        // the path needs, duplicates inside a read are found by looking back through the read.
        uint64_t *by_read = ha.p;
        if (h_info[2] == 1) {
            const uint32_t n_a = h_info[3], n_b = (uint32_t)(n_hits - n_a);
            const uint32_t n_tiles = ceil_div_u64(n_hits, kMergeTile);
            DevBuf<uint32_t> part;
            KG_ALLOC(ctx, part, (size_t)n_tiles + 1);
            KG_LAUNCH(ctx, merge_partition_kernel, grid_for((uint64_t)n_tiles + 1, kThreads), kThreads, 0, ha.p, n_a, ha.p + n_a, n_b,
                      n_tiles, part.p);
            KG_LAUNCH(ctx, merge_runs_kernel, n_tiles, kThreads, 0, ha.p, n_a, ha.p + n_a, n_b, part.p, hb.p);
            by_read = hb.p;
        }
        // compaction needs a third buffer only when the merge used both: the packed input is dead after the merge,
        // but a read that is too long sends us back to it, so keep it and compact into scratch
        uint64_t *dst = by_read == ha.p ? hb.p : nullptr;
        if (!dst) { KG_ALLOC(ctx, hp->hc, n_hits); dst = hp->hc.p; }
        KG_TRY((device_scan<uint32_t>(ctx, n_hits, FirstInReadFlag{by_read, info.p + 4}, CompactKeysU64{by_read, dst}, d_cnt.p)));
        uint32_t too_long = 0;
        KG_TRY(read_back(ctx, info.p + 4, &too_long, 1));
        if (!too_long) {
            KG_TRY(read_back(ctx, d_cnt.p, &n_uniq, 1));
            grouped = true;
            other = dst;
        }
    }
    if (!grouped) {
        int np = plan_radix_passes(0, bn, 32, 32 + bits_for(h_info[0]), passes);
        KG_TRY(radix_sort_u64(ctx, ha.p, hb.p, n_hits, passes, np, &sorted));
        other = sorted == ha.p ? hb.p : ha.p;
        KG_TRY((device_scan<uint32_t>(ctx, n_hits, HeadFlagU64{sorted}, CompactKeysU64{sorted, other}, d_cnt.p)));
        KG_TRY(read_back(ctx, d_cnt.p, &n_uniq, 1));
    }
    const uint64_t *hits = other;  // unique hits grouped by read (sorted when the general path ran), n_uniq of them
    hp->hits = hits;
    st->n_unique_hits = n_uniq;
    // the segment scan below carries two 32-bit counters in one word whose top two bits are the scan's status flags
    if (n_uniq >= (1u << 31)) return ctx_fail(ctx, KOMBGPU_EINVAL, "%u distinct (read, unitig) hits exceed the 2^31 per-device limit", n_uniq);

    // 2. reads with >= 2 unitigs -> segments; pairs per segment -> offsets
    DevBuf<uint64_t> d_tot(ctx, 1);
    KG_ALLOC(ctx, hp->seg_head, (size_t)n_uniq / 2 + 1);
    KG_ALLOC(ctx, hp->seg_tail, (size_t)n_uniq / 2 + 1);
    if (!d_tot) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
    KG_TRY((device_scan<uint64_t>(ctx, n_uniq, SegFlagIn{hits, n_uniq}, SegFlagOut{hp->seg_head.p, hp->seg_tail.p}, d_tot.p)));
    uint64_t seg_tot = 0;
    KG_TRY(read_back(ctx, d_tot.p, &seg_tot, 1));
    hp->n_seg = (uint32_t)(seg_tot >> 32);
    KG_ALLOC(ctx, hp->seg_base, (size_t)hp->n_seg + 1);
    KG_TRY((device_scan<uint64_t>(ctx, hp->n_seg, SegPairsIn{hp->seg_head.p, hp->seg_tail.p}, SegPairsOut{hp->seg_base.p}, d_tot.p)));
    KG_TRY(read_back(ctx, d_tot.p, &hp->n_pairs, 1));
    st->n_pairs = hp->n_pairs;
    return KOMBGPU_OK;
}

int pack_pairs(kombgpu_ctx *ctx, const uint32_t *u, const uint32_t *v, uint64_t n, uint32_t n_vertices, uint64_t *dst) {
    DevBuf<uint32_t> info(ctx, 2);
    if (!info) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
    KG_CUDA(ctx, cudaMemsetAsync(info.p, 0, 2 * sizeof(uint32_t), ctx->stream));
    if (n) KG_LAUNCH(ctx, pack_pairs_kernel, min(grid_for(n, kThreads), 148u * 16u), kThreads, 0, u, v, n, n_vertices, dst, info.p);
    uint32_t h_info[2] = {0, 0};
    KG_TRY(read_back(ctx, info.p, h_info, 2));
    if (h_info[1]) return ctx_fail(ctx, KOMBGPU_EINVAL, "edge endpoint >= n_vertices (%u)", n_vertices);
    return KOMBGPU_OK;
}

int hits_to_edges(kombgpu_ctx *ctx, const uint32_t *read_key, const uint32_t *unitig, uint64_t n_hits, uint32_t n_vertices,
                  DevBuf<uint64_t> &edges, uint64_t *n_edges, kombgpu_stats *st, DevBuf<uint32_t> *mult, uint32_t *n_chunks) {
    DevBuf<uint64_t> pa, pb;
    uint64_t *psorted = nullptr;
    {
        HitPairs hp;
        KG_TRY(count_hit_pairs(ctx, read_key, unitig, n_hits, n_vertices, &hp, st));
        const uint64_t n_pairs = hp.n_pairs;
        const int bn = bits_for(n_vertices > 0 ? n_vertices - 1 : 0);
        if (const uint64_t chunk = pair_chunk(n_pairs)) {
            // 3'. chunks of pairs, each emitted from its global pair index
            EdgeSink sink{&edges, n_edges, mult, n_chunks};
            return chunked_edges(ctx, n_pairs, chunk, bn, [&](uint64_t p0, uint64_t p1, uint64_t *dst) { return hp.emit(p0, p1, dst); },
                                 &sink);
        }
        if (n_pairs >= (1ull << 32))
            return ctx_fail(ctx, KOMBGPU_EINVAL, "%llu clique pairs exceed the 2^32 per-device limit", (unsigned long long)n_pairs);

        // 3. emit all pairs, sort
        KG_ALLOC(ctx, pa, n_pairs);
        KG_ALLOC(ctx, pb, n_pairs);
        psorted = pa.p;
        if (n_pairs) {
            KG_TRY(hp.emit(0, n_pairs, pa.p));
            RadixPass passes[8];
            const int np = plan_radix_passes(0, bn, 32, 32 + bn, passes);
            KG_TRY(radix_sort_u64(ctx, pa.p, pb.p, n_pairs, passes, np, &psorted));
        }
    }   // the hits and segments are dead
    if (n_chunks) *n_chunks = 1;
    return unique_edges(ctx, psorted, st->n_pairs, edges, n_edges, mult);
}

int pairs_to_edges(kombgpu_ctx *ctx, const uint32_t *u, const uint32_t *v, uint64_t n_pairs, uint32_t n_vertices,
                   DevBuf<uint64_t> &edges, uint64_t *n_edges, DevBuf<uint32_t> *mult, uint32_t *n_chunks) {
    if (const uint64_t chunk = pair_chunk(n_pairs)) {
        // chunks of the input, packed and range-checked as the one-shot path does
        auto emit = [&](uint64_t p0, uint64_t p1, uint64_t *dst) { return pack_pairs(ctx, u + p0, v + p0, p1 - p0, n_vertices, dst); };
        EdgeSink sink{&edges, n_edges, mult, n_chunks};
        return chunked_edges(ctx, n_pairs, chunk, bits_for(n_vertices > 0 ? n_vertices - 1 : 0), emit, &sink);
    }
    if (n_chunks) *n_chunks = 1;
    DevBuf<uint64_t> ka, kb;
    uint64_t *sorted = nullptr;
    KG_TRY(pairs_to_sorted_keys(ctx, u, v, n_pairs, n_vertices, ka, kb, &sorted));
    return unique_edges(ctx, sorted, n_pairs, edges, n_edges, mult);
}

int row_starts(kombgpu_ctx *ctx, const uint64_t *keys, uint64_t count, uint32_t base, uint32_t n_rows, uint32_t lo_bound, uint32_t *start,
               uint32_t *err_dev) {
    // a gap longer than kGapShort rows is recorded: at most n_rows / kGapShort + 1 of them
    DevBuf<RowGap> gaps;
    DevBuf<uint32_t> n_gaps(ctx, 1);
    KG_ALLOC(ctx, gaps, (size_t)n_rows / (size_t)kGapShort + 2);
    if (!n_gaps) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
    KG_CUDA(ctx, cudaMemsetAsync(n_gaps.p, 0, sizeof(uint32_t), ctx->stream));
    KG_LAUNCH(ctx, row_bounds_kernel, min(grid_for(count + 1, kThreads), 148u * 16u), kThreads, 0, keys, count, base, n_rows, lo_bound, start,
              gaps.p, n_gaps.p, err_dev);
    KG_LAUNCH(ctx, row_gaps_kernel, 148u * 4u, kThreads, 0, gaps.p, n_gaps.p, start);
    return KOMBGPU_OK;
}

int forward_index(kombgpu_ctx *ctx, const uint64_t *edges, uint64_t E, uint32_t n, uint32_t **fwd_start_out) {
    DevBuf<uint32_t> fwd_start;
    KG_ALLOC(ctx, fwd_start, (size_t)n + 1);
    KG_TRY(row_starts(ctx, edges, E, 0u, n, 0xffffffffu, fwd_start.p, nullptr));
    *fwd_start_out = fwd_start.take();
    return KOMBGPU_OK;
}

// unique simple edges (sorted, u < v) -> CSR of the symmetric graph
int csr_from_edges(kombgpu_ctx *ctx, DevBuf<uint64_t> &edges, uint64_t E, uint32_t n, kombgpu_graph *g) {
    g->n = n;
    g->n_edges = E;
    g->st.n_edges = E;
    g->st.n_vertices = n;
    DevBuf<uint64_t> sw_a, sw_b;
    uint64_t *swapped = nullptr;
    KG_TRY(swapped_sorted(ctx, edges.p, E, n, sw_a, sw_b, &swapped));
    DevBuf<uint32_t> back_start;
    KG_ALLOC(ctx, back_start, (size_t)n + 1);
    if (!g->fwd_start) KG_TRY(forward_index(ctx, edges.p, E, n, &g->fwd_start));   // kept: the CSR form of the edge list
    const uint32_t *fwd_start_p = g->fwd_start;
    KG_TRY(row_starts(ctx, swapped, E, 0u, n, 0xffffffffu, back_start.p, nullptr));

    DevBuf<uint64_t> row_ptr;
    DevBuf<int32_t> deg, max_deg(ctx, 1);
    DevBuf<uint32_t> col;
    KG_ALLOC(ctx, row_ptr, (size_t)n + 1);
    KG_ALLOC(ctx, deg, n);
    KG_ALLOC(ctx, col, 2 * E);
    if (!max_deg) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
    KG_CUDA(ctx, cudaMemsetAsync(max_deg.p, 0, sizeof(int32_t), ctx->stream));
    KG_TRY((device_scan<uint64_t>(ctx, n, DegreeIn{fwd_start_p, back_start.p}, DegreeOut{row_ptr.p, deg.p},
                                  (uint64_t *)nullptr)));
    if (n) KG_LAUNCH(ctx, reduce_max_i32_kernel, min(grid_for(n, kThreads), 148u * 8u), kThreads, 0, deg.p, (uint64_t)n, max_deg.p);
    KG_LAUNCH(ctx, set_u64_kernel, 1, 1, 0, row_ptr.p + n, 2 * E);
    if (E)
        KG_LAUNCH(ctx, fill_col_kernel, min(grid_for(E, kThreads), 148u * 16u), kThreads, 0, edges.p, swapped, E, row_ptr.p,
                  fwd_start_p, back_start.p, col.p);
    KG_TRY(read_back(ctx, max_deg.p, &g->st.max_degree, 1));
    g->edges = edges.take();
    g->row_ptr = row_ptr.take();
    g->col = col.take();
    g->deg = deg.take();
    return KOMBGPU_OK;
}

// directed entries (src << 32 | dst) with src in [v_lo, v_lo + n_local), any order, duplicates allowed
// -> CSR rows of this rank: row_ptr[n_local + 1], col[] = global ids (every row ascending), deg[]
int csr_from_directed(kombgpu_ctx *ctx, const uint64_t *entries, uint64_t count, uint32_t v_lo, uint32_t n_local,
                      uint32_t n_global, uint64_t **row_ptr_out, uint32_t **col_out, int32_t **deg_out, int32_t *max_deg_out,
                      uint64_t *n_directed_out) {
    if (count >= (1ull << 32)) return ctx_fail(ctx, KOMBGPU_EINVAL, "more than 2^32 directed entries on one device");
    const int bn = bits_for(n_global > 0 ? n_global - 1 : 0);
    DevBuf<uint64_t> ka, kb, uniq;
    KG_ALLOC(ctx, ka, count);
    KG_ALLOC(ctx, kb, count);
    uint64_t *sorted = ka.p;
    if (count) {
        KG_CUDA(ctx, cudaMemcpyAsync(ka.p, entries, count * sizeof(uint64_t), cudaMemcpyDeviceToDevice, ctx->stream));
        RadixPass passes[8];
        int np = plan_radix_passes(0, bn, 32, 32 + bn, passes);
        KG_TRY(radix_sort_u64(ctx, ka.p, kb.p, count, passes, np, &sorted));
    }
    DevBuf<uint32_t> d_count(ctx, 1);
    if (!d_count) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
    KG_ALLOC(ctx, uniq, count);
    KG_TRY((device_scan<uint32_t>(ctx, count, AnyHeadFlag{sorted}, CompactKeysU64{sorted, uniq.p}, d_count.p)));
    uint32_t nd32 = 0;
    KG_TRY(read_back(ctx, d_count.p, &nd32, 1));
    const uint64_t nd = nd32;
    DevBuf<uint64_t> row_ptr;
    DevBuf<uint32_t> col;
    DevBuf<int32_t> deg, max_deg(ctx, 1);
    KG_ALLOC(ctx, row_ptr, (size_t)n_local + 1);
    KG_ALLOC(ctx, col, nd);
    KG_ALLOC(ctx, deg, n_local);
    if (!max_deg) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
    KG_CUDA(ctx, cudaMemsetAsync(max_deg.p, 0, sizeof(int32_t), ctx->stream));
    DevBuf<uint32_t> d_err(ctx, 1);
    if (!d_err) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
    KG_CUDA(ctx, cudaMemsetAsync(d_err.p, 0, sizeof(uint32_t), ctx->stream));
    KG_LAUNCH(ctx, row_bounds_base_kernel, min(grid_for(nd + 1, kThreads), 148u * 16u), kThreads, 0, uniq.p, nd, v_lo, n_local,
              n_global ? n_global : 1u, row_ptr.p, d_err.p);
    uint32_t h_err = 0;
    KG_TRY(read_back(ctx, d_err.p, &h_err, 1));
    if (h_err) return ctx_fail(ctx, KOMBGPU_EINVAL, "a directed entry lies outside this rank's rows [%u, %u) or names a unitig >= %u", v_lo, v_lo + n_local, n_global);
    if (nd) KG_LAUNCH(ctx, part_cols_kernel, min(grid_for(nd, kThreads), 148u * 16u), kThreads, 0, uniq.p, nd, col.p);
    if (n_local)
        KG_LAUNCH(ctx, part_degree_kernel, min(grid_for(n_local, kThreads), 148u * 8u), kThreads, 0, row_ptr.p, n_local, deg.p,
                  max_deg.p);
    KG_TRY(read_back(ctx, max_deg.p, max_deg_out, 1));
    *n_directed_out = nd;
    *row_ptr_out = row_ptr.take();
    *col_out = col.take();
    *deg_out = deg.take();
    return KOMBGPU_OK;
}

// copy an existing CSR (device) into a graph; degrees from the row lengths
int adopt_csr(kombgpu_ctx *ctx, const uint64_t *row_ptr, const uint32_t *col, uint32_t n, kombgpu_graph *g) {
    uint64_t n_dir = 0;
    KG_TRY(read_back(ctx, row_ptr + n, &n_dir, 1));
    if (n_dir && !col) return ctx_fail(ctx, KOMBGPU_EINVAL, "null col array");
    DevBuf<uint64_t> rp;
    DevBuf<uint32_t> cl;
    DevBuf<int32_t> deg, max_deg(ctx, 1);
    KG_ALLOC(ctx, rp, (size_t)n + 1);
    KG_ALLOC(ctx, cl, n_dir);
    KG_ALLOC(ctx, deg, n);
    if (!max_deg) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
    KG_CUDA(ctx, cudaMemcpyAsync(rp.p, row_ptr, ((size_t)n + 1) * sizeof(uint64_t), cudaMemcpyDeviceToDevice, ctx->stream));
    if (n_dir) KG_CUDA(ctx, cudaMemcpyAsync(cl.p, col, n_dir * sizeof(uint32_t), cudaMemcpyDeviceToDevice, ctx->stream));
    KG_CUDA(ctx, cudaMemsetAsync(max_deg.p, 0, sizeof(int32_t), ctx->stream));
    if (n) KG_LAUNCH(ctx, part_degree_kernel, min(grid_for(n, kThreads), 148u * 8u), kThreads, 0, rp.p, n, deg.p, max_deg.p);
    KG_TRY(read_back(ctx, max_deg.p, &g->st.max_degree, 1));
    g->n = n;
    g->n_edges = n_dir / 2;
    g->st.n_vertices = n;
    g->st.n_edges = n_dir / 2;
    g->row_ptr = rp.take();
    g->col = cl.take();
    g->deg = deg.take();
    return KOMBGPU_OK;
}

int build_from_pairs(kombgpu_ctx *ctx, const uint32_t *u, const uint32_t *v, uint64_t n_pairs, uint32_t n_vertices,
                     kombgpu_graph *g) {
    DevBuf<uint64_t> edges;
    uint64_t E = 0;
    g->st.n_pairs = n_pairs;
    DevBuf<uint32_t> mult;
    KG_TRY(pairs_to_edges(ctx, u, v, n_pairs, n_vertices, edges, &E, &mult, &g->build_chunks));
    g->mult = mult.take();
    return csr_from_edges(ctx, edges, E, n_vertices, g);
}

int build_from_hits(kombgpu_ctx *ctx, const uint32_t *read_key, const uint32_t *unitig, uint64_t n_hits,
                    uint32_t n_vertices, kombgpu_graph *g) {
    DevBuf<uint64_t> edges;
    uint64_t E = 0;
    DevBuf<uint32_t> mult;
    KG_TRY(hits_to_edges(ctx, read_key, unitig, n_hits, n_vertices, edges, &E, &g->st, &mult, &g->build_chunks));
    g->mult = mult.take();
    return csr_from_edges(ctx, edges, E, n_vertices, g);
}

void graph_release(kombgpu_graph *g) {
    if (!g || !g->ctx) return;
    kombgpu_ctx *ctx = g->ctx;
    truss_release(g);
    format_release(g);
    if (g->edges) ws_free(ctx, g->edges);
    if (g->fwd_start) ws_free(ctx, g->fwd_start);
    if (g->mult) ws_free(ctx, g->mult);
    g->fwd_start = nullptr; g->mult = nullptr;
    if (g->row_ptr) ws_free(ctx, g->row_ptr);
    if (g->col) ws_free(ctx, g->col);
    if (g->deg) ws_free(ctx, g->deg);
    if (g->core) ws_free(ctx, g->core);
    if (g->score) ws_free(ctx, g->score);
    g->edges = nullptr; g->row_ptr = nullptr; g->col = nullptr; g->deg = nullptr; g->core = nullptr; g->score = nullptr;
}

}  // namespace kg
