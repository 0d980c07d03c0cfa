// pcore.cu — the graph analyses of the partitioned graph: the maximal core with the trussness of its edges (the
// reference's Kgraph::runTruss, truss.cu) and the densest k-core (densest.cu), which consume the finished coreness,
// and the densest block (densest.cu), which needs only the build.
//
// The first two need the coreness of unitigs other ranks own (the far end of an edge).  Every rank puts its coreness slice into
// the symmetric heap and pulls the others' with plain device-to-device copies, as rpeel.cu pulls rows: 4 bytes per
// unitig of the graph cross a link, once per call.
//   truss    every rank selects the maximal core over all ids (max_coreness is global), filters and relabels ITS slice
//            of the canonical edge list and pulls the other ranks' filtered slices.  The relabelling is monotone and the
//            slices are in u-range order, so their concatenation is the canonical sorted edge list of the maximal core:
//            no sort.  Every rank then runs the single-GPU truss on it (replicated, like rpeel.cu), so the maximal core
//            has to fit one GPU and hold fewer than 2^32 edges; the whole graph need not.
//   densest  every rank counts its unitigs per coreness and its forward edges per min(core(u), core(v)); the summed
//            histograms go through the selection of the single-GPU densest core.
//   block    the single-GPU pass loop (densest_block_passes) with steps that span the ranks: each rank marks its own
//            unitigs and lists the removed global ids in the symmetric heap, every rank pulls the lists of the pass
//            (4 bytes per removed unitig cross a link, n_global x 4 bytes over the whole call) and lowers the degrees
//            of its own survivors, through the layout the build left (grouped by neighbour: push; rows: pull).  Two
//            exchanges per pass sum the counts in rank order, so every rank holds the same totals and threshold.
// Every exchange carries each rank's status: a failure on one rank (allocation, CUDA) makes every rank return an error
// at the next exchange, the failing rank its own and the others that of the first failing rank.
#include <cstring>
#include <vector>

#include "dgraph.cuh"
#include "kombgpu_debug.h"

namespace kg {
namespace {

// rank q owns ids [*lo, *lo + rows)
uint32_t rows_of(const kombgpu_dist_graph *g, int q, uint64_t *lo) {
    *lo = (uint64_t)q * g->step;
    if (*lo >= g->n_global) return 0u;
    const uint64_t hi = *lo + g->step < g->n_global ? *lo + g->step : g->n_global;
    return (uint32_t)(hi - *lo);
}

int cuda_rc(kombgpu_ctx *ctx, cudaError_t e, const char *what) {
    return e == cudaSuccess ? KOMBGPU_OK : ctx_fail(ctx, KOMBGPU_ECUDA, "%s: %s", what, cudaGetErrorString(e));
}

// comm_exchange of k words per rank (out[q * k + j]) that also carries every rank's status `rc`
int exchange_rc(kombgpu_comm *c, int rc, const unsigned long long *vals, int k, unsigned long long *out) {
    unsigned long long mine[kCtlWords], all[kMaxRanks * kCtlWords];
    mine[0] = rc != KOMBGPU_OK ? (unsigned long long)-rc : 0ull;
    for (int j = 0; j < k; ++j) mine[1 + j] = vals[j];
    KG_TRY(comm_exchange(c, mine, k + 1, all));
    for (int q = 0; q < c->world; ++q)
        for (int j = 0; j < k; ++j) out[q * k + j] = all[q * (k + 1) + 1 + j];
    if (rc != KOMBGPU_OK) return rc;   // this rank's own message stands
    for (int q = 0; q < c->world; ++q)
        if (all[q * (k + 1)]) return ctx_fail(c->ctx, -(int)all[q * (k + 1)], "rank %d failed; the call stopped on every rank", q);
    return KOMBGPU_OK;
}

int barrier_rc(kombgpu_comm *c, int rc) { return exchange_rc(c, rc, nullptr, 0, nullptr); }

// core_all[x] = coreness of unitig x, for every unitig of the graph
int gather_coreness(kombgpu_dist_graph *g, DevBuf<int32_t> &core_all) {
    kombgpu_comm *c = g->comm;
    kombgpu_ctx *ctx = g->ctx;
    SymRewind heap{c, sym_mark(c)};
    int32_t *mine = nullptr;
    PeerPtrs<int32_t> peers{};
    KG_TRY(sym_alloc(c, (size_t)g->step, &mine, &peers));   // the same size on every rank
    int rc = KOMBGPU_OK;
    if (!core_all.alloc(ctx, g->n_global)) rc = ctx_fail(ctx, KOMBGPU_ENOMEM, "the coreness of %u unitigs", g->n_global);
    if (rc == KOMBGPU_OK && g->n_local)
        rc = cuda_rc(ctx, cudaMemcpyAsync(mine, g->core, (size_t)g->n_local * sizeof(int32_t), cudaMemcpyDeviceToDevice, ctx->stream),
                     "coreness slice");
    KG_TRY(barrier_rc(c, rc));   // every rank's slice is in place
    for (int q = 0; q < c->world && rc == KOMBGPU_OK; ++q) {
        uint64_t lo = 0;
        const uint32_t rows = rows_of(g, q, &lo);
        if (rows)
            rc = cuda_rc(ctx, cudaMemcpyAsync(core_all.p + lo, peers.p[q], (size_t)rows * sizeof(int32_t), cudaMemcpyDeviceToDevice, ctx->stream),
                         "coreness slice of a peer");
    }
    return barrier_rc(c, rc);   // everybody has read every slice: the buffer may go
}

unsigned long long double_bits(double d) {
    unsigned long long b;
    memcpy(&b, &d, sizeof b);
    return b;
}

double bits_double(unsigned long long b) {
    double d;
    memcpy(&d, &b, sizeof d);
    return d;
}

// ---- densest block

// the ids removed in pass t, gathered from every rank: pass_all[x] = t
__global__ void __launch_bounds__(kBlockThreads) block_scatter_kernel(const uint32_t *__restrict__ ids, uint32_t n, uint32_t t,
                                                                      uint32_t *__restrict__ pass_all) {
    for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) pass_all[ids[k]] = t;
}

// grouped by neighbour (nbr_ptr / nbr): one warp per removed unitig x walks this rank's neighbours of x (local ids)
__global__ void __launch_bounds__(kBlockThreads) block_push_kernel(const uint32_t *__restrict__ nbr_ptr, const uint32_t *__restrict__ nbr,
                                                                   const uint32_t *__restrict__ ids, uint32_t n_ids, uint32_t t,
                                                                   const uint32_t *__restrict__ pass, int32_t *__restrict__ deg_s,
                                                                   BlockPass *__restrict__ st) {
    block_update_warps(nbr_ptr, nbr, ids, n_ids, t, pass, deg_s, st);
}

constexpr uint32_t kPullChunk = 1024;   // row entries per warp task: a longer row (a hub) is shared by several warps

// rows (row_ptr32 / col): every warp takes kPullChunk consecutive entries of the rank's rows.  For each row u they
// overlap whose unitig survives or left in pass t, it counts the neighbours that left in pass t (pass_all): a survivor
// loses them (single), a unitig of the same pass counts them in `both`.  Rows cut by a chunk boundary are combined by
// the atomics on deg_s; every value here is uniform over the warp.
__global__ void __launch_bounds__(kBlockThreads) block_pull_kernel(const uint32_t *__restrict__ row_ptr, const uint32_t *__restrict__ col,
                                                                   uint32_t n_rows, uint32_t t, const uint32_t *__restrict__ pass,
                                                                   const uint32_t *__restrict__ pass_all, int32_t *__restrict__ deg_s,
                                                                   BlockPass *__restrict__ st) {
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5, lane = lane_id();
    const uint32_t n_entries = row_ptr[n_rows];
    unsigned long long single = 0, both = 0;
    for (uint64_t c0 = (uint64_t)warp * kPullChunk; c0 < n_entries; c0 += (uint64_t)n_warps * kPullChunk) {
        const uint32_t e0 = (uint32_t)c0, e1 = (uint32_t)min(c0 + kPullChunk, (uint64_t)n_entries);
        uint32_t lo = 0, hi = n_rows;   // the first row that ends after e0
        while (lo < hi) {
            const uint32_t mid = (lo + hi) >> 1;
            if (row_ptr[mid + 1] > e0) hi = mid;
            else lo = mid + 1;
        }
        for (uint32_t u = lo; u < n_rows; ++u) {
            const uint32_t r0 = row_ptr[u];
            if (r0 >= e1) break;
            const uint32_t pu = pass[u];
            if (pu != kBlockUnset && pu != t) continue;
            const uint32_t a = max(r0, e0), b = min(row_ptr[u + 1], e1);
            uint32_t cnt = 0;
            for (uint32_t e = a; e < b; e += 32) {
                const bool hit = lane < b - e && pass_all[col[e + lane]] == t;
                cnt += __popc(__ballot_sync(kFullMask, hit));
            }
            if (cnt && lane == 0) {
                if (pu == kBlockUnset) {
                    atomicSub(&deg_s[u], (int32_t)cnt);
                    single += cnt;
                } else {
                    both += cnt;
                }
            }
        }
    }
    if (lane == 0) {
        if (single) atomicAdd(&st->single, single);
        if (both) atomicAdd(&st->both, both);
    }
}

// The steps of one pass on the partitioned graph.  mark: each rank marks its slice and lists the removed global ids in
// the symmetric heap; the exchange that follows carries every rank's status, removed count and removed weight, summed
// in rank order, so every rank holds the same totals.  update: every rank pulls the lists of the pass, its survivors
// lose the removed neighbours, and the second exchange sums `single` and `both` (and is the barrier after which the
// lists may be written again).
struct DistBlockSteps final : BlockSteps {
    kombgpu_dist_graph *g;
    kombgpu_comm *c;
    kombgpu_ctx *ctx;
    const double *w = nullptr;
    DevBuf<double> w_dev;
    DevBuf<int32_t> deg_s;
    DevBuf<uint32_t> pass, ids, pass_all;   // pass: [n_local]; ids: [n_global] one pass's removed ids; pass_all: [n_global], rows only
    DevBuf<BlockPass> st;
    uint32_t *list = nullptr;               // [step] this rank's list, in the symmetric heap
    PeerPtrs<uint32_t> lists{};
    unsigned long long removed[kMaxRanks] = {};   // per rank, in the current pass
    explicit DistBlockSteps(kombgpu_dist_graph *gr) : g(gr), c(gr->comm), ctx(gr->ctx) {}

    // everything before the first exchange: checks, workspace, the copy of the degrees and this rank's weight sum
    int prepare(const double *weight, int use_scores, double eps, double *W) {
        const uint32_t n = g->n_local;
        *W = 0.0;
        if (!(eps >= 0.0) || eps > 1e6) return ctx_fail(ctx, KOMBGPU_EINVAL, "eps must be in [0, 1e6]");
        if (weight && use_scores) return ctx_fail(ctx, KOMBGPU_EINVAL, "give weights or ask for the CORE-A scores, not both");
        if (use_scores && !g->has_score) return ctx_fail(ctx, KOMBGPU_ESTATE, "the CORE-A scores have not been computed");
        if (weight)
            for (uint32_t i = 0; i < n; ++i) {
                if (!(weight[i] >= 0.0) || weight[i] > 1e300) return ctx_fail(ctx, KOMBGPU_EINVAL, "weights must be finite and >= 0");
                *W += weight[i];
            }
        KG_ALLOC(ctx, deg_s, n);
        KG_ALLOC(ctx, pass, n);
        KG_ALLOC(ctx, ids, g->n_global);
        KG_ALLOC(ctx, st, 1);
        KG_CUDA(ctx, cudaMemsetAsync(pass.p, 0xff, (size_t)(n ? n : 1) * sizeof(uint32_t), ctx->stream));
        if (n) KG_CUDA(ctx, cudaMemcpyAsync(deg_s.p, g->deg, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToDevice, ctx->stream));
        if (g->peel_choice != 0) {
            KG_ALLOC(ctx, pass_all, g->n_global);
            KG_CUDA(ctx, cudaMemsetAsync(pass_all.p, 0xff, (size_t)(g->n_global ? g->n_global : 1) * sizeof(uint32_t), ctx->stream));
        }
        if (weight && n) {
            KG_ALLOC(ctx, w_dev, n);
            KG_CUDA(ctx, cudaMemcpyAsync(w_dev.p, weight, (size_t)n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
            w = w_dev.p;
        }
        if (use_scores) {
            w = g->score;
            KG_TRY(block_weight_sum(ctx, w, deg_s.p, n, list, st.p, W));
        }
        return KOMBGPU_OK;
    }

    int mark_local(double thr, uint32_t t, BlockPass *mine) {
        KG_CUDA(ctx, cudaMemsetAsync(st.p, 0, sizeof(BlockPass), ctx->stream));
        KG_LAUNCH(ctx, block_mark_kernel, block_grid(ctx, g->n_local), kBlockThreads, 0, w, deg_s.p, g->n_local, thr, t, g->v_lo, pass.p, list,
                  st.p);
        return read_back(ctx, st.p, mine, 1);
    }

    int mark(double thr, uint32_t t, BlockPass *h) override {
        BlockPass mine{};
        const int rc = mark_local(thr, t, &mine);
        unsigned long long v[2] = {mine.removed, double_bits(mine.w_removed)}, all[kMaxRanks * 2];
        KG_TRY(exchange_rc(c, rc, v, 2, all));
        *h = BlockPass{};
        for (int q = 0; q < c->world; ++q) {
            removed[q] = all[2 * q];
            h->removed += all[2 * q];
            h->w_removed += bits_double(all[2 * q + 1]);
        }
        return KOMBGPU_OK;
    }

    int update_local(uint32_t t, BlockPass *mine) {
        uint64_t n_ids = 0;
        for (int q = 0; q < c->world; ++q) {
            if (removed[q])
                KG_CUDA(ctx, cudaMemcpyAsync(ids.p + n_ids, lists.p[q], removed[q] * sizeof(uint32_t), cudaMemcpyDeviceToDevice, ctx->stream));
            n_ids += removed[q];
        }
        KG_CUDA(ctx, cudaMemsetAsync(st.p, 0, sizeof(BlockPass), ctx->stream));
        if (g->peel_choice == 0) {
            if (!n_ids) return read_back(ctx, st.p, mine, 1);
            const uint32_t grid = min(ceil_div_u64(n_ids * 32u, kBlockThreads), (uint32_t)ctx->sm_count * 16u);
            KG_LAUNCH(ctx, block_push_kernel, grid, kBlockThreads, 0, g->nbr_ptr, g->nbr, ids.p, (uint32_t)n_ids, t, pass.p, deg_s.p, st.p);
        } else {
            KG_LAUNCH(ctx, block_scatter_kernel, block_grid(ctx, n_ids), kBlockThreads, 0, ids.p, (uint32_t)n_ids, t, pass_all.p);
            if (g->n_directed) {
                const uint32_t grid = min(ceil_div_u64(ceil_div_u64(g->n_directed, kPullChunk) * 32ull, kBlockThreads), (uint32_t)ctx->sm_count * 16u);
                KG_LAUNCH(ctx, block_pull_kernel, grid, kBlockThreads, 0, g->row_ptr32, g->col, g->n_local, t, pass.p, pass_all.p, deg_s.p, st.p);
            }
        }
        return read_back(ctx, st.p, mine, 1);
    }

    int update(uint32_t t, BlockPass *h) override {
        BlockPass mine{};
        const int rc = update_local(t, &mine);
        unsigned long long v[2] = {mine.single, mine.both}, all[kMaxRanks * 2];
        KG_TRY(exchange_rc(c, rc, v, 2, all));
        h->single = h->both = 0;
        for (int q = 0; q < c->world; ++q) {
            h->single += all[2 * q];
            h->both += all[2 * q + 1];
        }
        return KOMBGPU_OK;
    }
};

}  // namespace

int dist_max_core_truss(kombgpu_dist_graph *g) {
    kombgpu_comm *c = g->comm;
    kombgpu_ctx *ctx = g->ctx;
    const int world = c->world;
    truss_free(ctx, &g->tr);
    g->has_truss = false;
    EvTimer timer(ctx);

    // 1. the coreness of every unitig, and with it the maximal core over all ids, relabelled in order
    DevBuf<int32_t> core_all;
    KG_TRY(gather_coreness(g, core_all));
    g->ms_truss[0] = timer.lap();
    DevBuf<uint32_t> sub_id, core_vid;
    uint32_t n_core = 0;
    int rc = max_core_vertices(ctx, core_all.p, g->n_global, g->st.max_coreness, sub_id, core_vid, &n_core);
    core_all.release();
    // 2. this rank's slice of the induced edges
    DevBuf<uint64_t> slice;
    uint64_t m_mine = 0;
    if (rc == KOMBGPU_OK) rc = max_core_edges(ctx, g->edges, g->n_fwd, sub_id.p, slice, &m_mine);
    sub_id.release();

    // 3. every rank's slice, in rank order: the canonical sorted edge list of the maximal core
    unsigned long long cnt = m_mine, all_cnt[kMaxRanks];
    KG_TRY(exchange_rc(c, rc, &cnt, 1, all_cnt));
    uint64_t off[kMaxRanks + 1] = {}, max_cnt = 0;
    for (int q = 0; q < world; ++q) {
        off[q + 1] = off[q] + all_cnt[q];
        max_cnt = all_cnt[q] > max_cnt ? all_cnt[q] : max_cnt;
    }
    const uint64_t m = off[world];
    if (m >= (1ull << 32))
        return ctx_fail(ctx, KOMBGPU_EINVAL, "the maximal core has %llu edges: its truss is computed on one GPU and needs fewer than 2^32",
                        (unsigned long long)m);
    DevBuf<uint64_t> sub_edges;
    {
        SymRewind heap{c, sym_mark(c)};
        uint64_t *mine = nullptr;
        PeerPtrs<uint64_t> peers{};
        KG_TRY(sym_alloc(c, (size_t)max_cnt, &mine, &peers));
        if (m_mine)
            rc = cuda_rc(ctx, cudaMemcpyAsync(mine, slice.p, m_mine * sizeof(uint64_t), cudaMemcpyDeviceToDevice, ctx->stream), "edge slice");
        if (rc == KOMBGPU_OK && !sub_edges.alloc(ctx, m))
            rc = ctx_fail(ctx, KOMBGPU_ENOMEM, "the %llu edges of the maximal core", (unsigned long long)m);
        KG_TRY(barrier_rc(c, rc));   // every rank's slice is in place
        slice.release();
        for (int q = 0; q < world && rc == KOMBGPU_OK; ++q)
            if (all_cnt[q])
                rc = cuda_rc(ctx, cudaMemcpyAsync(sub_edges.p + off[q], peers.p[q], all_cnt[q] * sizeof(uint64_t), cudaMemcpyDeviceToDevice,
                                                  ctx->stream), "edge slice of a peer");
        KG_TRY(barrier_rc(c, rc));   // everybody has read every slice: the buffers may go
    }
    g->ms_truss[1] = timer.lap();

    // 4. the truss of the whole maximal core, on every rank; one answer on every rank
    rc = barrier_rc(c, sub_edges_truss(ctx, sub_edges, m, core_vid, n_core, &g->tr));
    g->ms_truss[2] = timer.lap();
    if (rc != KOMBGPU_OK) {
        truss_free(ctx, &g->tr);
        return rc;
    }
    g->has_truss = true;
    return KOMBGPU_OK;
}

int dist_densest_core(kombgpu_dist_graph *g, DensestCore *out) {
    kombgpu_comm *c = g->comm;
    kombgpu_ctx *ctx = g->ctx;
    const int world = c->world;
    const uint64_t n = g->n_global, n_edges = g->n_edges_global;
    const uint32_t n_bins = n && n_edges ? (uint32_t)g->st.max_coreness + 1 : 0u;   // the same on every rank
    std::vector<unsigned long long> h(2 * (size_t)n_bins, 0ull);
    if (n_bins) {
        DevBuf<int32_t> core_all;
        KG_TRY(gather_coreness(g, core_all));
        SymRewind heap{c, sym_mark(c)};
        unsigned long long *mine = nullptr;
        PeerPtrs<unsigned long long> peers{};
        KG_TRY(sym_alloc(c, 2 * (size_t)n_bins, &mine, &peers));
        // unitigs per coreness over the local slice; forward edges per min(core(u), core(v)) over the local edges
        int rc = cuda_rc(ctx, cudaMemsetAsync(mine, 0, 2 * (size_t)n_bins * sizeof(unsigned long long), ctx->stream), "histograms");
        if (rc == KOMBGPU_OK) rc = level_histogram(ctx, g->core, nullptr, g->n_local, n_bins, mine);
        if (rc == KOMBGPU_OK) rc = level_histogram(ctx, core_all.p, g->edges, g->n_fwd, n_bins, mine + n_bins);
        KG_TRY(barrier_rc(c, rc));   // every rank's histograms are in place
        core_all.release();
        DevBuf<unsigned long long> all;
        std::vector<unsigned long long> h_all((size_t)world * 2 * n_bins);
        if (!all.alloc(ctx, h_all.size())) rc = ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
        for (int q = 0; q < world && rc == KOMBGPU_OK; ++q)
            rc = cuda_rc(ctx, cudaMemcpyAsync(all.p + (size_t)q * 2 * n_bins, peers.p[q], 2 * (size_t)n_bins * sizeof(unsigned long long),
                                              cudaMemcpyDeviceToDevice, ctx->stream), "histograms of a peer");
        if (rc == KOMBGPU_OK) rc = read_back(ctx, all.p, h_all.data(), h_all.size());
        KG_TRY(barrier_rc(c, rc));   // everybody has read every histogram: the buffer may go
        for (int q = 0; q < world; ++q)
            for (size_t i = 0; i < h.size(); ++i) h[i] += h_all[(size_t)q * 2 * n_bins + i];
    }
    *out = densest_level(h.data(), h.data() + n_bins, n_bins, n, n_edges);
    return KOMBGPU_OK;
}

int dist_densest_block(kombgpu_dist_graph *g, const double *weight, int use_scores, double eps, DensestBlock *out, uint8_t *member) {
    kombgpu_comm *c = g->comm;
    kombgpu_ctx *ctx = g->ctx;
    SymRewind heap{c, sym_mark(c)};
    DistBlockSteps steps(g);
    KG_TRY(sym_alloc(c, (size_t)g->step, &steps.list, &steps.lists));   // the same size on every rank
    // the first exchange: every rank's status, eps, mode and weight sum
    double W_mine = 0.0;
    const int rc = steps.prepare(weight, use_scores, eps, &W_mine);
    unsigned long long v[3] = {double_bits(eps), (unsigned long long)(use_scores != 0), double_bits(W_mine)}, all[kMaxRanks * 3];
    KG_TRY(exchange_rc(c, rc, v, 3, all));
    double W = 0.0;
    for (int q = 0; q < c->world; ++q) {
        if (all[3 * q] != v[0]) return ctx_fail(ctx, KOMBGPU_EINVAL, "eps differs between the ranks");
        if (all[3 * q + 1] != v[1]) return ctx_fail(ctx, KOMBGPU_EINVAL, "use_scores differs between the ranks");
        W += bits_double(all[3 * q + 2]);
    }
    KG_TRY(densest_block_passes(ctx, g->n_global, g->n_edges_global, W, eps, steps, out));
    return block_member(ctx, steps.pass.p, g->n_local, out->t_best, member);
}

}  // namespace kg

using namespace kg;

extern "C" {

int kombgpu_dist_max_core_truss(kombgpu_dist_graph *g, uint32_t *n_core_vertices, uint64_t *n_core_edges, int32_t *max_trussness,
                                uint32_t *n_truss_vertices) {
    if (!g) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = g->ctx;
    if (!g->has_core) return ctx_fail(ctx, KOMBGPU_ESTATE, "kombgpu_dist_max_core_truss needs kombgpu_dist_coreness first");
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    if (!g->has_truss) KG_TRY(dist_max_core_truss(g));
    if (n_core_vertices) *n_core_vertices = g->tr.n_core;
    if (n_core_edges) *n_core_edges = g->tr.m;
    if (max_trussness) *max_trussness = g->tr.tmax;
    if (n_truss_vertices) *n_truss_vertices = g->tr.n_vertices;
    return KOMBGPU_OK;
}

int kombgpu_dist_max_core_edges(const kombgpu_dist_graph *g, uint32_t *u, uint32_t *v, int32_t *trussness) {
    if (!g) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = g->ctx;
    if (!g->has_truss) return ctx_fail(ctx, KOMBGPU_ESTATE, "call kombgpu_dist_max_core_truss first");
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    return truss_edges_to_host(ctx, g->tr, u, v, trussness);
}

int kombgpu_dist_truss_vertices(const kombgpu_dist_graph *g, uint32_t *vids) {
    if (!g) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = g->ctx;
    if (!g->has_truss) return ctx_fail(ctx, KOMBGPU_ESTATE, "call kombgpu_dist_max_core_truss first");
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    return truss_vertices_to_host(ctx, g->tr, vids);
}

int kombgpu_dist_densest_core(kombgpu_dist_graph *g, int32_t *k_star, uint32_t *n_vertices, uint64_t *n_edges, double *density) {
    if (!g) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = g->ctx;
    if (!g->has_core) return ctx_fail(ctx, KOMBGPU_ESTATE, "kombgpu_dist_densest_core needs kombgpu_dist_coreness first");
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    DensestCore best{};
    KG_TRY(dist_densest_core(g, &best));
    if (k_star) *k_star = best.k;
    if (n_vertices) *n_vertices = (uint32_t)best.n_vertices;
    if (n_edges) *n_edges = best.n_edges;
    if (density) *density = best.density;
    return KOMBGPU_OK;
}

int kombgpu_dist_densest_block(kombgpu_dist_graph *g, const double *weight, int use_scores, double eps, uint32_t *n_vertices,
                               uint64_t *n_edges, double *weight_sum, double *density, uint32_t *n_passes, uint8_t *member) {
    if (!g) return KOMBGPU_EINVAL;
    KG_CUDA(g->ctx, cudaSetDevice(g->ctx->device));
    DensestBlock best{};
    KG_TRY(dist_densest_block(g, weight, use_scores, eps, &best, member));
    if (n_vertices) *n_vertices = (uint32_t)best.n_vertices;
    if (n_edges) *n_edges = best.n_edges;
    if (weight_sum) *weight_sum = best.weight_sum;
    if (density) *density = best.density;
    if (n_passes) *n_passes = best.passes;
    return KOMBGPU_OK;
}

// measurement aid (include/kombgpu_debug.h): the CUDA-event split of the last kombgpu_dist_max_core_truss on this rank
int kombgpu_debug_dist_truss_timing(const kombgpu_dist_graph *g, float *ms_core_gather, float *ms_slice_gather, float *ms_truss) {
    if (!g) return KOMBGPU_EINVAL;
    if (!g->has_truss) return ctx_fail(g->ctx, KOMBGPU_ESTATE, "call kombgpu_dist_max_core_truss first");
    if (ms_core_gather) *ms_core_gather = g->ms_truss[0];
    if (ms_slice_gather) *ms_slice_gather = g->ms_truss[1];
    if (ms_truss) *ms_truss = g->ms_truss[2];
    return KOMBGPU_OK;
}

}  // extern "C"
