// pbuild.cu — stage 1 over the ranks of a communicator: the unitig graph partitioned by unitig-id range.
//
// Same reference steps as build.cu (getEdgeInfo + generateGraph + igraph_create + igraph_simplify,
// src/graph.cpp:259-285, 287-393, 418, 438); what is new is WHERE each step runs:
//   every rank    hits of its own reads -> clique pairs (min << 32 | max), unsorted
//   route 1       a pair goes to the rank that owns min: the scatter kernel ranks a tile by owner in shared memory
//                 and stores each owner's run straight into that rank's receive buffer (peer memory, NVLink) --
//                 bucketing and sending are one pass, and every pair is sorted exactly once, by its owner
//   owner         radix sort + adjacent-unique (+ multiplicities) -> its slice of the canonical edge list
//   route 2       (v - v_lo(owner(v))) << 32 | u of every edge goes to the owner of v
//   owner         forward and backward entries together, keyed by the NEIGHBOUR and sorted on it: for every unitig x of
//                 the graph the list of local unitigs adjacent to x -- the form the partitioned peel walks (ppeel.cu)
// The only host round trips are the two count exchanges (the receive sizes have to be known to allocate).
#include <cstdlib>

#include "dgraph.cuh"
#include "primitives.cuh"

namespace kg {
namespace {

constexpr int kThreads = 256;
constexpr int kRtThreads = 256;
constexpr int kRtItems = 8;
constexpr int kRtTile = kRtThreads * kRtItems;
constexpr int kRtWarps = kRtThreads / 32;

inline uint32_t grid_for(uint64_t n, int per_block) { return ceil_div_u64(n ? n : 1, per_block); }

// counts[o] += number of keys whose owner (hi word / step) is o
__global__ void __launch_bounds__(kRtThreads) route_count_kernel(const uint64_t *__restrict__ keys, uint64_t n, uint32_t step, int world,
                                                                 unsigned long long *__restrict__ counts, uint32_t *__restrict__ err) {
    __shared__ uint32_t s_cnt[kMaxRanks];
    if (threadIdx.x < kMaxRanks) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    const uint32_t lane = lane_id();
    for (uint64_t base = (uint64_t)blockIdx.x * kRtTile; base < n; base += (uint64_t)gridDim.x * kRtTile) {
#pragma unroll
        for (int j = 0; j < kRtItems; ++j) {
            const uint64_t i = base + (uint64_t)j * kRtThreads + threadIdx.x;
            uint32_t o = 0xffffffffu;
            if (i < n) {
                o = (uint32_t)(keys[i] >> 32) / step;
                if (o >= (uint32_t)world) { atomicExch(err, 1u); o = 0xffffffffu; }
            }
            const uint32_t same = __match_any_sync(kFullMask, o);
            if (o != 0xffffffffu && lane == (uint32_t)__ffs(same) - 1u) atomicAdd(&s_cnt[o], (uint32_t)__popc(same));
        }
    }
    __syncthreads();
    if (threadIdx.x < world && s_cnt[threadIdx.x]) atomicAdd(&counts[threadIdx.x], (unsigned long long)s_cnt[threadIdx.x]);
}

struct RouteSmem {
    uint64_t keys[kRtTile];
    uint32_t warp_cnt[kRtWarps][kMaxRanks];
    uint32_t local_start[kMaxRanks + 1];      // first slot of owner o inside the staged tile
    unsigned long long global_base[kMaxRanks];   // position of that slot in owner o's receive buffer
};

// One tile: rank the keys by owner (warp match + per-warp counters), reserve a run in every owner's receive buffer
// with one atomic per owner, stage the tile in owner order, store each run contiguously into peer memory.
__global__ void __launch_bounds__(kRtThreads) route_scatter_kernel(const uint64_t *__restrict__ keys, uint64_t n, uint32_t step, int world,
                                                                   bool rebase, unsigned long long *cursors, PeerPtrs<uint64_t> dst) {
    __shared__ RouteSmem s;
    const uint32_t warp = threadIdx.x >> 5, lane = lane_id();
    for (uint64_t base = (uint64_t)blockIdx.x * kRtTile; base < n; base += (uint64_t)gridDim.x * kRtTile) {
        for (int i = threadIdx.x; i < kRtWarps * kMaxRanks; i += kRtThreads) (&s.warp_cnt[0][0])[i] = 0;
        __syncthreads();
        uint64_t key[kRtItems];
        uint32_t own[kRtItems], rank[kRtItems];
        // warp-striped: item j of lane l is element warp * 256 + j * 32 + l
        const uint32_t warp_base = warp * (32 * kRtItems);
#pragma unroll
        for (int j = 0; j < kRtItems; ++j) {
            const uint64_t i = base + warp_base + j * 32 + lane;
            own[j] = 0xffffffffu;
            key[j] = 0;
            if (i < n) {
                key[j] = keys[i];
                const uint32_t hi = (uint32_t)(key[j] >> 32);
                const uint32_t o = min(hi / step, (uint32_t)world - 1u);   // out-of-range ids were rejected by the count pass
                own[j] = o;
                if (rebase) key[j] = ((uint64_t)(hi - o * step) << 32) | (uint32_t)key[j];
            }
        }
#pragma unroll
        for (int j = 0; j < kRtItems; ++j) {
            const uint32_t same = __match_any_sync(kFullMask, own[j]);
            const uint32_t lead = (uint32_t)__ffs(same) - 1u;
            uint32_t b = 0;
            if (own[j] != 0xffffffffu && lane == lead) b = atomicAdd(&s.warp_cnt[warp][own[j]], (uint32_t)__popc(same));
            rank[j] = __shfl_sync(kFullMask, b, lead) + __popc(same & lanemask_lt());
        }
        __syncthreads();
        if (threadIdx.x < (uint32_t)world) {   // per owner: exclusive prefix over the warps, total
            uint32_t run = 0;
            for (int w = 0; w < kRtWarps; ++w) {
                const uint32_t c = s.warp_cnt[w][threadIdx.x];
                s.warp_cnt[w][threadIdx.x] = run;
                run += c;
            }
            s.local_start[threadIdx.x + 1] = run;   // totals for now
            s.global_base[threadIdx.x] = run ? atomicAdd(&cursors[threadIdx.x], (unsigned long long)run) : 0ull;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t run = 0;
            s.local_start[0] = 0;
            for (int o = 0; o < world; ++o) { const uint32_t c = s.local_start[o + 1]; s.local_start[o + 1] = run + c; run += c; }
        }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < kRtItems; ++j)
            if (own[j] != 0xffffffffu) s.keys[s.local_start[own[j]] + s.warp_cnt[warp][own[j]] + rank[j]] = key[j];
        __syncthreads();
        const uint32_t count = s.local_start[world];
        for (uint32_t i = threadIdx.x; i < count; i += kRtThreads) {
            int o = 0;
            while (i >= s.local_start[o + 1]) ++o;
            dst.p[o][s.global_base[o] + (i - s.local_start[o])] = s.keys[i];
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(kThreads) swap_edges_kernel(const uint64_t *__restrict__ edges, uint64_t n, uint64_t *__restrict__ out) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t e = edges[i];
        out[i] = (e << 32) | (e >> 32);
    }
}

// the local adjacency entries keyed by the neighbour: entry i < n_fwd is the forward edge (u, v) -> (v << 32 | u - v_lo);
// entry n_fwd + j is arrival j ((u - v_lo) << 32 | w) -> (w << 32 | u - v_lo), and counts one backward neighbour of u
// by_row: the keys are (u - v_lo) << 32 | neighbour instead (the rank's rows, for the asynchronous peel)
__global__ void __launch_bounds__(kThreads) nbr_keys_kernel(const uint64_t *__restrict__ edges, uint64_t n_fwd, const uint64_t *__restrict__ back,
                                                            uint64_t n_back, uint32_t v_lo, uint32_t n_local, uint32_t n_global, bool by_row,
                                                            uint64_t *__restrict__ keys, uint32_t *__restrict__ err) {
    const uint64_t total = n_fwd + n_back;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t u, w;
        if (i < n_fwd) {
            const uint64_t e = edges[i];
            u = (uint32_t)(e >> 32) - v_lo;
            w = (uint32_t)e;
        } else {
            const uint64_t s = back[i - n_fwd];
            u = (uint32_t)(s >> 32);
            w = (uint32_t)s;
            if (u >= n_local || w >= n_global) { atomicExch(err, 2u); keys[i] = 0; continue; }   // a mis-routed entry must not write past the arrays
        }
        keys[i] = by_row ? (((uint64_t)u << 32) | w) : (((uint64_t)w << 32) | u);
    }
}

// back_cnt[u] += 1 for every arrival ((u - v_lo) << 32 | w): the backward neighbours of the local unitigs
__global__ void __launch_bounds__(kThreads) back_count_kernel(const uint64_t *__restrict__ back, uint64_t n_back, uint32_t n_local, uint32_t n_global,
                                                              int32_t *__restrict__ back_cnt, uint32_t *__restrict__ err) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_back; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t s = back[i];
        const uint32_t u = (uint32_t)(s >> 32), w = (uint32_t)s;
        if (u >= n_local || w >= n_global) { atomicExch(err, 2u); continue; }
        atomicAdd(&back_cnt[u], 1);
    }
}

// deg[u] = forward neighbours (from the forward index) + backward neighbours (counted by back_count_kernel)
__global__ void __launch_bounds__(kThreads) pdegree_kernel(const uint32_t *__restrict__ fwd_start, uint32_t n_local, int32_t *__restrict__ deg,
                                                           int32_t *__restrict__ max_deg) {
    int32_t m = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_local; i += (uint64_t)gridDim.x * blockDim.x) {
        const int32_t d = deg[i] + (int32_t)(fwd_start[i + 1] - fwd_start[i]);
        deg[i] = d;
        m = max(m, d);
    }
    m = warp_reduce_max(m);
    if (lane_id() == 0 && m) atomicMax(max_deg, m);
}

__global__ void __launch_bounds__(kThreads) low_words_kernel(const uint64_t *__restrict__ keys, uint64_t n, uint32_t *__restrict__ out) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) out[i] = (uint32_t)keys[i];
}

// key (col[e] << 32 | u) for every entry e of local row u: the rows keyed by neighbour
__global__ void __launch_bounds__(kThreads) row_keys_kernel(const uint32_t *__restrict__ row_ptr, const uint32_t *__restrict__ col, uint32_t n_local,
                                                            uint64_t n, uint64_t *__restrict__ keys) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t lo = 0, hi = n_local;   // the last row that starts at or before i
        while (hi - lo > 1) {
            const uint32_t mid = (lo + hi) >> 1;
            if (row_ptr[mid] <= i) lo = mid; else hi = mid;
        }
        keys[i] = ((uint64_t)col[i] << 32) | lo;
    }
}

}  // namespace

// KOMBGPU_DIST_PEEL = async | log | auto (default).  The asynchronous peel (apeel.cu) decrements a neighbour where it
// lives, with an atomic over NVLink: a hub unitig takes one remote atomic per neighbour, all on one address, and those
// serialise at its home L2 (measured on 8 GPUs: cfg3, R-MAT with hubs of 10^5 .. 6 x 10^5 neighbours, 85 ms against 52 ms
// for the log-based peel; cfg2 x 8, largest hub 1.7 x 10^5, 13.0 against 14.4 ms; a 1/8 share of cfg4, degrees <= 55, 6.7
// against 14.7 ms).  Its walk is also the simpler, slower one per entry (a system-scope atomic and an owner lookup per
// neighbour): cfg4 at full size, 243 M adjacency entries per rank and only 28 levels, takes it 42.9 ms against 23.9 ms;
// a 1/8 share of cfg4 on 2 GPUs (122 M entries per rank) 22.1 against 15.0 ms; cfg2 (66 M per rank) 9.2 against 11.1 ms.
// auto: asynchronous unless the largest degree of the graph exceeds kAsyncMaxDegree, or a rank holds more than
// kAsyncMaxEntries adjacency entries of a FLAT graph (largest degree <= kFlatDegree, hence few levels and short chains:
// the peel is then bound by the rate of decrements, not by the length of its chains).
constexpr int32_t kAsyncMaxDegree = 1 << 18;
constexpr int32_t kFlatDegree = 1024;
constexpr unsigned long long kAsyncMaxEntries = 96ull << 20;
// A graph small enough for one GPU to peel in a few milliseconds is not partitioned for the peel at all (rpeel.cu): every
// rank pulls the other ranks' rows and runs the single-GPU kernel (cfg2 x 2 / x 4: 4.4 / 10.9 ms against 9.3 / 18.6 ms).
// Not beyond four ranks: on 8 GPUs the pull and the peel of the whole graph cost more than the partitioned peel's hops
// (cfg2 x 8: 21.5 against 12.7 ms; a 1/8 share of cfg4: 11.2 against 7.9 ms).
constexpr unsigned long long kReplicateMaxEntries = 300ull << 20;   // adjacency entries of the whole graph
constexpr int kReplicateMaxWorld = 4;
int dist_peel_mode() {   // 0 log, 1 async, 2 auto, 3 replicated
    const char *e = getenv("KOMBGPU_DIST_PEEL");
    if (e && e[0] == 'l') return 0;
    if (e && e[0] == 'a' && e[1] == 's') return 1;
    if (e && e[0] == 'r') return 3;
    return 2;
}

int route_keys(kombgpu_comm *c, const uint64_t *keys, uint64_t n, uint32_t step, bool rebase, uint64_t **recv, uint64_t *n_recv,
               int local_rc) {
    kombgpu_ctx *ctx = c->ctx;
    const int world = c->world;
    DevBuf<unsigned long long> d_counts(ctx, 2 * kMaxRanks);   // [counts | cursors]
    DevBuf<uint32_t> d_err(ctx, 1);
    if (!d_counts || !d_err) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
    const uint32_t grid = min(grid_for(n, kRtTile), (uint32_t)ctx->sm_count * 8u);
    unsigned long long h_counts[kMaxRanks + 1] = {};
    uint32_t h_err = 0;
    if (local_rc == KOMBGPU_OK) {   // a rank that has failed already sends nothing and only reports its error
        KG_CUDA(ctx, cudaMemsetAsync(d_counts.p, 0, 2 * kMaxRanks * sizeof(unsigned long long), ctx->stream));
        KG_CUDA(ctx, cudaMemsetAsync(d_err.p, 0, sizeof(uint32_t), ctx->stream));
        if (n) KG_LAUNCH(ctx, route_count_kernel, grid, kRtThreads, 0, keys, n, step, world, d_counts.p, d_err.p);
        KG_TRY(read_back(ctx, d_counts.p, h_counts, kMaxRanks));
        KG_TRY(read_back(ctx, d_err.p, &h_err, 1));
    }
    // a rank with bad input still takes part in the exchange (its peers are waiting), then everybody fails together:
    // the error word is the rank's (negated) error code
    h_counts[world] = local_rc != KOMBGPU_OK ? (unsigned long long)-local_rc : (h_err ? (unsigned long long)-KOMBGPU_EINVAL : 0ull);
    unsigned long long matrix[kMaxRanks * (kMaxRanks + 1)];   // matrix[q * (world + 1) + p] = keys rank q sends to rank p
    KG_TRY(comm_exchange(c, h_counts, world + 1, matrix));
    unsigned long long my_off[kMaxRanks] = {}, max_recv = 0, mine = 0;
    for (int p = 0; p < world; ++p) {
        unsigned long long tot = 0;
        for (int q = 0; q < world; ++q) {
            if (q == c->rank) my_off[p] = tot;
            tot += matrix[q * (world + 1) + p];
        }
        if (tot > max_recv) max_recv = tot;
        if (p == c->rank) mine = tot;
    }
    for (int q = 0; q < world; ++q) {
        const unsigned long long e = matrix[q * (world + 1) + world];
        if (!e) continue;
        if (local_rc != KOMBGPU_OK) return local_rc;   // this rank's own message stands
        if (h_err) return ctx_fail(ctx, KOMBGPU_EINVAL, "a unitig id is outside [0, n_vertices_global) on some rank");
        return ctx_fail(ctx, -(int)e, "rank %d failed; the build stopped on every rank", q);
    }
    if (max_recv >= (1ull << 32)) return ctx_fail(ctx, KOMBGPU_EINVAL, "%llu keys routed to one rank exceed the 2^32 per-device limit", max_recv);
    uint64_t *buf = nullptr;
    PeerPtrs<uint64_t> peers{};
    KG_TRY(sym_alloc(c, (size_t)max_recv, &buf, &peers));
    KG_CUDA(ctx, cudaMemcpyAsync(d_counts.p + kMaxRanks, my_off, kMaxRanks * sizeof(unsigned long long), cudaMemcpyHostToDevice, ctx->stream));
    if (n) KG_LAUNCH(ctx, route_scatter_kernel, grid, kRtThreads, 0, keys, n, step, world, rebase, d_counts.p + kMaxRanks, peers);
    // everything every rank stored has landed once the exchange returns
    unsigned long long token = 1, tokens[kMaxRanks];
    KG_TRY(comm_exchange(c, &token, 1, tokens));
    *recv = buf;
    *n_recv = mine;
    return KOMBGPU_OK;
}

int dist_build(kombgpu_comm *c, const uint32_t *a, const uint32_t *b, uint64_t count, uint32_t n_global, bool from_hits,
               kombgpu_dist_graph *g) {
    kombgpu_ctx *ctx = c->ctx;
    const int world = c->world;
    if (n_global >= 0xfffffffeu) return ctx_fail(ctx, KOMBGPU_EINVAL, "n_vertices too large");
    g->comm = c;
    g->ctx = ctx;
    g->n_global = n_global;
    g->step = owner_step(n_global, world);
    const uint64_t lo64 = (uint64_t)c->rank * g->step, hi64 = lo64 + g->step;
    g->v_lo = (uint32_t)(lo64 < n_global ? lo64 : n_global);
    g->n_local = (uint32_t)((hi64 < n_global ? hi64 : n_global) - g->v_lo);
    g->st.n_global = n_global;
    g->st.v_lo = g->v_lo;
    g->st.n_local = g->n_local;
    g->st.max_coreness = -1;
    const uint32_t n_local = g->n_local;
    const int bn = bits_for(n_global > 0 ? n_global - 1 : 0);
    EvTimer total(ctx), split(ctx);

    // 1. count this rank's pairs (hits: unique hits, segments and their pair offsets) without emitting them
    HitPairs hp;
    uint64_t n_pairs = count;
    int rc_local = KOMBGPU_OK;
    if (from_hits) {
        kombgpu_stats st{};
        rc_local = count_hit_pairs(ctx, a, b, count, n_global, &hp, &st);
        n_pairs = hp.n_pairs;
        g->st.n_hits_local = count;
    }
    g->st.n_pairs_local = n_pairs;

    // one decision for every rank: one shot while the pairs of all ranks stay below 2^32 (so does every owner's share),
    // else R rounds of at most `chunk` pairs per rank (DESIGN.md §4).  A rank whose count failed reports its error here.
    unsigned long long mine_p[2] = {rc_local == KOMBGPU_OK ? n_pairs : 0ull, (unsigned long long)-rc_local}, all_p[kMaxRanks * 2];
    KG_TRY(comm_exchange(c, mine_p, 2, all_p));
    uint64_t sum_p = 0, max_p = 0;
    for (int q = 0; q < world; ++q) {
        sum_p += all_p[q * 2];
        max_p = all_p[q * 2] > max_p ? all_p[q * 2] : max_p;
    }
    if (rc_local != KOMBGPU_OK) return rc_local;
    for (int q = 0; q < world; ++q)
        if (all_p[q * 2 + 1]) return ctx_fail(ctx, -(int)all_p[q * 2 + 1], "rank %d failed; the build stopped on every rank", q);
    uint64_t chunk = 0;   // 0: one shot
    const uint64_t cap = pair_chunk_env();
    if (cap && max_p > cap) chunk = min(cap, (uint64_t)(0xffffffffu / (uint32_t)world));   // world x chunk < 2^32: an owner's counts are 32-bit
    else if (sum_p >= (1ull << 32)) chunk = kPairChunk / (uint64_t)world;   // an owner receives < 2^30 keys a round: bounds its buffers
    const uint64_t per_round = chunk ? chunk : n_pairs;
    const uint32_t rounds = chunk ? (uint32_t)((max_p + chunk - 1) / chunk) : 1u;
    g->build_rounds = rounds;

    // 2. every round: emit the next pairs, route them to the owner of min(u, v), sort there, then unique (one shot) or
    //    reduce and merge into the running edge list.  From here on a rank that fails keeps taking part in the
    //    exchanges, routes nothing and reports its error in the next route_keys, where every rank stops.
    SymRewind heap{c, sym_mark(c)};   // each round's receive buffer is released once it is reduced; all of them on failure
    if (chunk) {
        // an owner receives at most world x chunk keys a round: one segment of that size up front, so a round that
        // outgrows an earlier one does not stack another segment on the heap (same call on every rank: collective)
        uint64_t *reserve = nullptr;
        PeerPtrs<uint64_t> peers{};
        KG_TRY(sym_alloc(c, (size_t)(world * chunk), &reserve, &peers));
        sym_release(c, heap.mark);
    }
    DevBuf<uint64_t> edges, tmp;   // tmp: the sort's second buffer (in rounds also the reduced keys)
    DevBuf<uint32_t> mult, ccnt;   // ccnt: the reduced keys' counts
    // in rounds both are sized once for the largest receive, as the single-GPU chunk buffers are: no round reallocates
    if (chunk && (!tmp.alloc(ctx, world * chunk) || !ccnt.alloc(ctx, world * chunk)))
        rc_local = ctx_fail(ctx, KOMBGPU_ENOMEM, "device workspace for %llu routed pairs", (unsigned long long)(world * chunk));
    EdgeRun run;
    uint64_t n_fwd = 0, n_recv_total = 0;
    for (uint32_t r = 0; r < rounds; ++r) {
        const uint64_t p0 = min(n_pairs, (uint64_t)r * per_round), p1 = min(n_pairs, p0 + per_round);
        DevBuf<uint64_t> pairs;
        if (rc_local == KOMBGPU_OK) {
            if (!pairs.alloc(ctx, p1 - p0)) rc_local = ctx_fail(ctx, KOMBGPU_ENOMEM, "device workspace for %llu pairs", (unsigned long long)(p1 - p0));
            else rc_local = from_hits ? hp.emit(p0, p1, pairs.p) : pack_pairs(ctx, a + p0, b + p0, p1 - p0, n_global, pairs.p);
        }
        if (p1 >= n_pairs) hp.release();   // every pair of this rank is out: the hits and segments are dead
        uint64_t *recv = nullptr, n_recv = 0;
        KG_TRY(route_keys(c, pairs.p, rc_local == KOMBGPU_OK ? p1 - p0 : 0, g->step, false, &recv, &n_recv, rc_local));
        pairs.release();
        n_recv_total += n_recv;
        g->st.ms_build_route += split.lap();
        // route_keys succeeded, so no rank has failed so far
        rc_local = [&]() -> int {
            if (!chunk) KG_ALLOC(ctx, tmp, n_recv);
            RadixPass passes[8];
            const int np = plan_radix_passes(0, bn, 32, 32 + bn, passes);
            uint64_t *sorted = recv;
            KG_TRY(radix_sort_u64(ctx, recv, tmp.p, n_recv, passes, np, &sorted));
            if (!chunk) return unique_edges(ctx, sorted, n_recv, edges, &n_fwd, &mult);
            if (n_recv == 0) return KOMBGPU_OK;
            return merge_sorted_chunk(ctx, sorted, n_recv, sorted == recv ? tmp.p : recv, ccnt.p, &run);
        }();
        sym_release(c, heap.mark);   // the receive buffer is dead (stream-ordered: later kernels of this stream come after its readers)
        g->st.ms_build_sort += split.lap();
    }
    tmp.release();
    ccnt.release();
    if (chunk && rc_local == KOMBGPU_OK) {
        if (!run.keys && !run.keys.alloc(ctx, 0)) rc_local = ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
        if (!run.cnt && !run.cnt.alloc(ctx, 0)) rc_local = ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
        edges = std::move(run.keys);
        mult = std::move(run.cnt);
        n_fwd = run.n;
    }
    g->st.n_pairs_received = n_recv_total;
    g->n_fwd = n_fwd;
    g->st.n_fwd_local = n_fwd;

    // 3. reversed copies -> owner of max(u, v) (high word rebased to the owner's range); stable sort by row there
    DevBuf<uint64_t> swapped;
    if (rc_local == KOMBGPU_OK && !swapped.alloc(ctx, n_fwd)) rc_local = ctx_fail(ctx, KOMBGPU_ENOMEM, "device workspace for %llu edges", (unsigned long long)n_fwd);
    if (rc_local == KOMBGPU_OK && n_fwd)
        KG_LAUNCH(ctx, swap_edges_kernel, min(grid_for(n_fwd, kThreads), 148u * 16u), kThreads, 0, edges.p, n_fwd, swapped.p);
    uint64_t *back = nullptr, n_back = 0;
    KG_TRY(route_keys(c, swapped.p, rc_local == KOMBGPU_OK ? n_fwd : 0, g->step, true, &back, &n_back, rc_local));
    swapped.release();
    g->st.ms_build_route += split.lap();
    // 4. the local entries keyed by neighbour: (v << 32 | u - v_lo) for the forward edges, (w << 32 | u - v_lo) for what arrived;
    //    degrees from the forward index plus a count of the arrivals; one sort on the neighbour bits
    const uint64_t n_dir = n_fwd + n_back;
    if (n_dir >= (1ull << 32)) return ctx_fail(ctx, KOMBGPU_EINVAL, "%llu adjacency entries on one rank exceed the 2^32 per-device limit", (unsigned long long)n_dir);
    DevBuf<uint32_t> fwd_start, nbr_ptr, nbr, d_err(ctx, 1);
    DevBuf<int32_t> deg, max_deg(ctx, 1);
    DevBuf<uint64_t> keys_a, keys_b;
    KG_ALLOC(ctx, fwd_start, (size_t)n_local + 1);
    KG_ALLOC(ctx, deg, n_local);
    KG_ALLOC(ctx, keys_a, n_dir);
    KG_ALLOC(ctx, keys_b, n_dir);
    if (!d_err || !max_deg) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
    KG_CUDA(ctx, cudaMemsetAsync(d_err.p, 0, sizeof(uint32_t), ctx->stream));
    KG_CUDA(ctx, cudaMemsetAsync(max_deg.p, 0, sizeof(int32_t), ctx->stream));
    KG_CUDA(ctx, cudaMemsetAsync(deg.p, 0, (size_t)(n_local ? n_local : 1) * sizeof(int32_t), ctx->stream));
    KG_TRY(row_starts(ctx, edges.p, n_fwd, g->v_lo, n_local, n_global, fwd_start.p, d_err.p));
    // degrees first (forward index + a count of the arrivals): the largest one picks the peel, the peel picks the layout
    if (n_back)
        KG_LAUNCH(ctx, back_count_kernel, min(grid_for(n_back, kThreads), 148u * 16u), kThreads, 0, back, n_back, n_local, n_global, deg.p,
                  d_err.p);
    if (n_local)
        KG_LAUNCH(ctx, pdegree_kernel, min(grid_for(n_local, kThreads), 148u * 8u), kThreads, 0, fwd_start.p, n_local, deg.p, max_deg.p);
    int choice = dist_peel_mode() == 2 ? 0 : (dist_peel_mode() == 3 ? 2 : dist_peel_mode());
    if (dist_peel_mode() == 2) {   // the layout follows the peel, the peel follows the shape of the whole graph
        int32_t h_max_now = 0;
        KG_TRY(read_back(ctx, max_deg.p, &h_max_now, 1));
        unsigned long long mine_shape[2] = {(unsigned long long)(uint32_t)h_max_now, (unsigned long long)n_dir}, all_shape[kMaxRanks * 2];
        KG_TRY(comm_exchange(c, mine_shape, 2, all_shape));
        int32_t gmax_now = 0;
        unsigned long long dir_max = 0, dir_total = 0;
        for (int q = 0; q < world; ++q) {
            gmax_now = max(gmax_now, (int32_t)all_shape[q * 2]);
            dir_max = all_shape[q * 2 + 1] > dir_max ? all_shape[q * 2 + 1] : dir_max;
            dir_total += all_shape[q * 2 + 1];
        }
        if (world > 1 && world <= kReplicateMaxWorld && dir_total <= kReplicateMaxEntries) choice = 2;
        else choice = (gmax_now <= kAsyncMaxDegree && !(dir_max > kAsyncMaxEntries && gmax_now <= kFlatDegree)) ? 1 : 0;
    }
    const bool by_row = choice != 0;
    g->peel_choice = choice;
    if (n_dir)
        KG_LAUNCH(ctx, nbr_keys_kernel, min(grid_for(n_dir, kThreads), 148u * 16u), kThreads, 0, edges.p, n_fwd, back, n_back, g->v_lo, n_local,
                  n_global, by_row, keys_a.p, d_err.p);
    uint64_t *nsorted = keys_a.p;
    {
        RadixPass passes[8];
        const int np = plan_radix_passes(32, 32 + (by_row ? bits_for(n_local > 0 ? n_local - 1 : 0) : bn), 0, 0, passes);
        KG_TRY(radix_sort_u64(ctx, keys_a.p, keys_b.p, n_dir, passes, np, &nsorted));
    }
    g->st.ms_build_sort += split.lap();
    KG_ALLOC(ctx, nbr_ptr, (size_t)(by_row ? n_local : n_global) + 1);
    KG_ALLOC(ctx, nbr, n_dir);
    if (by_row) KG_TRY(row_starts(ctx, nsorted, n_dir, 0u, n_local, n_global ? n_global : 1u, nbr_ptr.p, d_err.p));
    else KG_TRY(row_starts(ctx, nsorted, n_dir, 0u, n_global, n_local ? n_local : 1u, nbr_ptr.p, d_err.p));
    if (n_dir) KG_LAUNCH(ctx, low_words_kernel, min(grid_for(n_dir, kThreads), 148u * 16u), kThreads, 0, nsorted, n_dir, nbr.p);
    uint32_t h_err = 0;
    int32_t h_max = 0;
    KG_TRY(read_back(ctx, d_err.p, &h_err, 1));
    KG_TRY(read_back(ctx, max_deg.p, &h_max, 1));
    keys_a.release();
    keys_b.release();
    sym_release(c, heap.mark);
    g->st.ms_build_csr = split.lap();

    // global figures (also the barrier that ends the stage: every rank's rows are complete)
    unsigned long long mine[4] = {n_fwd, (unsigned long long)(uint32_t)h_max, h_err, n_dir}, all[kMaxRanks * 4];
    KG_TRY(comm_exchange(c, mine, 4, all));
    uint64_t E = 0, sum_dir = 0;
    int32_t gmax = 0;
    bool bad = false;
    for (int q = 0; q < world; ++q) {
        E += all[q * 4];
        gmax = max(gmax, (int32_t)all[q * 4 + 1]);
        bad = bad || all[q * 4 + 2] != 0;
        sum_dir += all[q * 4 + 3];
    }
    if (bad) return ctx_fail(ctx, KOMBGPU_EINTERNAL, "a routed entry arrived at a rank that does not own its row");
    if (sum_dir != 2 * E) return ctx_fail(ctx, KOMBGPU_EINTERNAL, "directed entries (%llu) != 2 x edges (%llu)", (unsigned long long)sum_dir, (unsigned long long)(2 * E));
    g->n_directed = n_dir;
    g->n_edges_global = E;
    g->st.n_directed_local = n_dir;
    g->st.n_edges_global = E;
    g->st.max_degree = gmax;
    g->edges = edges.take();
    g->mult = mult.take();
    g->fwd_start = fwd_start.take();
    if (by_row) { g->row_ptr32 = nbr_ptr.take(); g->col = nbr.take(); }
    else { g->nbr_ptr = nbr_ptr.take(); g->nbr = nbr.take(); }
    g->deg = deg.take();
    g->st.ms_build = total.lap();
    return KOMBGPU_OK;
}

int dist_rows_to_nbr(kombgpu_dist_graph *g, DevBuf<uint32_t> &nbr_ptr, DevBuf<uint32_t> &nbr) {
    kombgpu_ctx *ctx = g->ctx;
    const uint64_t n_dir = g->n_directed;
    const uint32_t n_local = g->n_local, n_global = g->n_global;
    DevBuf<uint64_t> keys_a, keys_b;
    DevBuf<uint32_t> d_err(ctx, 1);
    if (!d_err) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
    KG_ALLOC(ctx, keys_a, n_dir);
    KG_ALLOC(ctx, keys_b, n_dir);
    KG_CUDA(ctx, cudaMemsetAsync(d_err.p, 0, sizeof(uint32_t), ctx->stream));
    if (n_dir) KG_LAUNCH(ctx, row_keys_kernel, min(grid_for(n_dir, kThreads), 148u * 16u), kThreads, 0, g->row_ptr32, g->col, n_local, n_dir, keys_a.p);
    // the sort, the row starts and the low words of dist_build's by-neighbour layout
    uint64_t *nsorted = keys_a.p;
    RadixPass passes[8];
    const int np = plan_radix_passes(32, 32 + bits_for(n_global > 0 ? n_global - 1 : 0), 0, 0, passes);
    KG_TRY(radix_sort_u64(ctx, keys_a.p, keys_b.p, n_dir, passes, np, &nsorted));
    KG_ALLOC(ctx, nbr_ptr, (size_t)n_global + 1);
    KG_ALLOC(ctx, nbr, n_dir);
    KG_TRY(row_starts(ctx, nsorted, n_dir, 0u, n_global, n_local ? n_local : 1u, nbr_ptr.p, d_err.p));
    if (n_dir) KG_LAUNCH(ctx, low_words_kernel, min(grid_for(n_dir, kThreads), 148u * 16u), kThreads, 0, nsorted, n_dir, nbr.p);
    uint32_t h_err = 0;
    KG_TRY(read_back(ctx, d_err.p, &h_err, 1));
    if (h_err) return ctx_fail(ctx, KOMBGPU_EINTERNAL, "the rows hold an entry outside the graph");
    return KOMBGPU_OK;
}

void dist_graph_release(kombgpu_dist_graph *g) {
    if (!g || !g->ctx) return;
    kombgpu_ctx *ctx = g->ctx;
    void *ptrs[] = {g->edges, g->mult, g->fwd_start, g->nbr_ptr, g->nbr, g->row_ptr32, g->col, g->deg, g->core, g->score};
    for (void *p : ptrs)
        if (p) ws_free(ctx, p);
    g->edges = nullptr; g->mult = nullptr; g->fwd_start = nullptr; g->nbr_ptr = nullptr; g->nbr = nullptr; g->row_ptr32 = nullptr; g->col = nullptr;
    g->deg = nullptr; g->core = nullptr; g->score = nullptr;
    truss_free(ctx, &g->tr);
    g->has_truss = false;
    dist_onion_release(g);
    dist_format_release(g);
}

}  // namespace kg
