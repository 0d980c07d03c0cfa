// densest.cu — densest k-core: the bulk analogue of the serial greedy densest-block peel the reference keeps
// (unreachable from main) in CombineCoreA::runMerge over HashIndexedMinHeap (src/CombineCoreA.h:45-219,
// src/HashIndexedMinHeap.h).  That code pops the minimum-priority node again and again, tracks
// density = (edges + suspiciousness left) / (nodes left) and returns the densest prefix of the removal order
// (Charikar's greedy 2-approximation run on a row copy and a column copy of every vertex; its tie order and an
// uninitialised `removed[]` make its exact output accidental, so it is not a parity target: SURVEY.md row A9).
// The peel this library already ran visits the same nested family of blocks level by level: the k-cores.  The
// densest of them is a 2-approximation of the densest subgraph as well (the ceil(rho*)-core is not empty and has
// minimum degree >= rho*), and it falls out of two histograms over the finished coreness array:
//   V_k = #{v : core(v) >= k},  E_k = #{(u,v) in E : min(core(u), core(v)) >= k},  density_k = E_k / V_k
// (the reference's suspSum / numNodes for suspiciousness == nullptr: 2 E_k directed entries over 2 V_k row+column
// nodes).  Among blocks of equal density the largest wins, as with the reference's strict `>` while it shrinks the
// block; k* is reported as the smallest coreness inside the block.
#include <vector>

#include "graph.cuh"

namespace kg {
namespace {

constexpr int kThreads = 256;
constexpr int kSmemBins = 4096;

// kEdges = false: hist[core[v]] += 1 over the `count` vertices; kEdges = true: hist[min(core[u], core[v])] += 1 over the
// `count` edges of the canonical edge list
template <bool kEdges>
__global__ void __launch_bounds__(kThreads) level_hist_kernel(const int32_t *__restrict__ core, const uint64_t *__restrict__ edges,
                                                              uint64_t count, uint32_t n_bins,
                                                              unsigned long long *__restrict__ hist) {
    __shared__ uint32_t s_hist[kSmemBins];
    const bool use_smem = n_bins <= kSmemBins;
    if (use_smem) {
        for (uint32_t i = threadIdx.x; i < n_bins; i += kThreads) s_hist[i] = 0;
        __syncthreads();
    }
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (uint64_t)gridDim.x * blockDim.x) {
        int32_t c;
        if (kEdges) {
            const uint64_t e = edges[i];
            c = min(core[(uint32_t)(e >> 32)], core[(uint32_t)e]);
        } else {
            c = core[i];
        }
        if (use_smem) atomicAdd(&s_hist[c], 1u);
        else atomicAdd(&hist[c], 1ull);
    }
    if (use_smem) {
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < n_bins; i += kThreads)
            if (s_hist[i]) atomicAdd(&hist[i], (unsigned long long)s_hist[i]);
    }
}

// ---- densest BLOCK: the reference's greedy peel itself (CombineCoreA::runMerge, src/CombineCoreA.h:45-219) in bulk form.
// runMerge keeps a row copy and a column copy of every unitig with priority = suspiciousness + degree towards the other
// copy's survivors (:56-93), removes the minimum again and again (:112-131), keeps suspiciousSum / nodes left as the
// density (:133-141) and lowers the neighbours' priorities (:147-172).  On a symmetric adjacency the two copies of a
// unitig always carry the same priority, so the peel is Charikar's greedy on the graph itself with
//     f(S) = sum_{v in S} w(v) + |E(S)|,   density(S) = f(S) / |S|,   priority(v) = w(v) + deg_S(v).
// One node per step is a serial algorithm; the bulk form (Bahmani, Kumar, Vassilvitskii 2012) removes, per pass, EVERY
// survivor with priority <= 2 (1 + eps) density(S): the priorities sum to at most 2 f(S), so a pass removes at least an
// eps / (1 + eps) share of the survivors (O(log n / eps) passes) and the best S seen is a 2 (1 + eps)-approximation,
// against 2 for the serial order.  Ties need no rule: a pass is a set.

// one warp per removed unitig: its survivors lose a neighbour
__global__ void __launch_bounds__(kThreads) block_update_kernel(const uint64_t *__restrict__ row_ptr, const uint32_t *__restrict__ col,
                                                                const uint32_t *__restrict__ list, uint32_t n_list,
                                                                uint32_t t, const uint32_t *__restrict__ pass, int32_t *__restrict__ deg_s,
                                                                BlockPass *__restrict__ st) {
    block_update_warps(row_ptr, col, list, n_list, t, pass, deg_s, st);
}

// the single-GPU steps: every unitig is local, the list holds the removed ids
struct GraphBlockSteps final : BlockSteps {
    kombgpu_ctx *ctx;
    const kombgpu_graph *g;
    const double *w;
    int32_t *deg_s;
    uint32_t *pass, *list;
    BlockPass *st;
    GraphBlockSteps(kombgpu_ctx *c, const kombgpu_graph *gr, const double *wt, int32_t *d, uint32_t *p, uint32_t *l, BlockPass *s)
        : ctx(c), g(gr), w(wt), deg_s(d), pass(p), list(l), st(s) {}
    int mark(double thr, uint32_t t, BlockPass *h) override {
        KG_CUDA(ctx, cudaMemsetAsync(st, 0, sizeof(BlockPass), ctx->stream));
        KG_LAUNCH(ctx, block_mark_kernel, block_grid(ctx, g->n), kBlockThreads, 0, w, deg_s, g->n, thr, t, 0u, pass, list, st);
        return read_back(ctx, st, h, 1);
    }
    int update(uint32_t t, BlockPass *h) override {
        const uint32_t ugrid = min(ceil_div_u64(h->removed * 32u, kThreads), (uint32_t)ctx->sm_count * 16u);
        KG_LAUNCH(ctx, block_update_kernel, ugrid, kThreads, 0, g->row_ptr, g->col, list, (uint32_t)h->removed, t, pass, deg_s, st);
        return read_back(ctx, st, h, 1);
    }
};

}  // namespace

__global__ void __launch_bounds__(kBlockThreads) block_mark_kernel(const double *__restrict__ w, const int32_t *__restrict__ deg_s, uint32_t n,
                                                                   double thr, uint32_t t, uint32_t id_base, uint32_t *__restrict__ pass,
                                                                   uint32_t *__restrict__ list, BlockPass *__restrict__ st) {
    double wsum = 0.0;
    for (uint32_t base = blockIdx.x * blockDim.x; base < n; base += gridDim.x * blockDim.x) {
        const uint32_t i = base + threadIdx.x;
        bool take = false;
        if (i < n && pass[i] == kBlockUnset) {
            const double wi = w ? w[i] : 0.0;
            take = wi + (double)deg_s[i] <= thr;
            if (take) { pass[i] = t; wsum += wi; }
        }
        const uint32_t m = __ballot_sync(kFullMask, take);
        if (m) {
            uint32_t pos = 0;
            if (lane_id() == 0) pos = (uint32_t)atomicAdd(&st->removed, (unsigned long long)__popc(m));
            pos = __shfl_sync(kFullMask, pos, 0) + __popc(m & lanemask_lt());
            if (take) list[pos] = id_base + i;
        }
    }
    wsum = warp_reduce_add(wsum);
    if (lane_id() == 0 && wsum != 0.0) atomicAdd(&st->w_removed, wsum);
}

__global__ void __launch_bounds__(kBlockThreads) block_member_kernel(const uint32_t *__restrict__ pass, uint32_t n, uint32_t t_best,
                                                                     uint8_t *__restrict__ member) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) member[i] = pass[i] >= t_best ? 1 : 0;
}

int block_weight_sum(kombgpu_ctx *ctx, const double *w, const int32_t *deg_s, uint32_t n, uint32_t *list, BlockPass *st, double *sum) {
    *sum = 0.0;
    if (!n) return KOMBGPU_OK;
    DevBuf<uint32_t> scratch;
    KG_ALLOC(ctx, scratch, n);
    KG_CUDA(ctx, cudaMemsetAsync(st, 0, sizeof(BlockPass), ctx->stream));
    KG_CUDA(ctx, cudaMemsetAsync(scratch.p, 0xff, (size_t)n * sizeof(uint32_t), ctx->stream));
    KG_LAUNCH(ctx, block_mark_kernel, block_grid(ctx, n), kBlockThreads, 0, w, deg_s, n, 1e308, 0u, 0u, scratch.p, list, st);
    BlockPass h{};
    KG_TRY(read_back(ctx, st, &h, 1));
    *sum = h.w_removed;
    return KOMBGPU_OK;
}

int block_member(kombgpu_ctx *ctx, const uint32_t *pass, uint32_t n, uint32_t t_best, uint8_t *member) {
    if (!member || !n) return KOMBGPU_OK;
    DevBuf<uint8_t> member_dev;
    KG_ALLOC(ctx, member_dev, n);
    KG_LAUNCH(ctx, block_member_kernel, block_grid(ctx, n), kBlockThreads, 0, pass, n, t_best, member_dev.p);
    KG_CUDA(ctx, cudaMemcpyAsync(member, member_dev.p, n, cudaMemcpyDeviceToHost, ctx->stream));
    KG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return KOMBGPU_OK;
}

int densest_block_passes(kombgpu_ctx *ctx, uint64_t n, uint64_t n_edges, double W, double eps, BlockSteps &steps, DensestBlock *out) {
    uint64_t E = n_edges, N = n;
    DensestBlock best{n, n_edges, W, n ? (W + (double)E) / (double)n : 0.0, 0u, 0u};
    uint32_t t = 0;
    while (N > 0) {
        const double rho = (W + (double)E) / (double)N;
        if (t == 0 || rho > best.density) best = DensestBlock{N, E, W, rho, 0u, t};
        double thr = 2.0 * (1.0 + eps) * rho;
        BlockPass h{};
        for (int attempt = 0;; ++attempt) {
            KG_TRY(steps.mark(thr, t, &h));
            if (h.removed) break;
            // the smallest priority is at most the mean, which is at most 2 rho; only rounding in the weight sums can leave a pass empty
            if (attempt >= 60) return ctx_fail(ctx, KOMBGPU_EINTERNAL, "densest block: a pass removed nothing");
            thr = thr * 1.0000001 + 1e-300;
        }
        KG_TRY(steps.update(t, &h));
        N -= h.removed;
        E -= h.single + h.both / 2;
        W -= h.w_removed;
        if (W < 0.0 || N == 0) W = 0.0;
        ++t;
        if (t == kBlockUnset - 1) return ctx_fail(ctx, KOMBGPU_EINTERNAL, "densest block: too many passes");
    }
    best.passes = t;
    *out = best;
    return KOMBGPU_OK;
}

int level_histogram(kombgpu_ctx *ctx, const int32_t *core, const uint64_t *edges, uint64_t count, uint32_t n_bins,
                    unsigned long long *hist) {
    if (count == 0) return KOMBGPU_OK;
    const uint32_t grid = min(ceil_div_u64(count, kThreads), (uint32_t)ctx->sm_count * 8u);
    if (edges) KG_LAUNCH(ctx, level_hist_kernel<true>, grid, kThreads, 0, core, edges, count, n_bins, hist);
    else KG_LAUNCH(ctx, level_hist_kernel<false>, grid, kThreads, 0, core, (const uint64_t *)nullptr, count, n_bins, hist);
    return KOMBGPU_OK;
}

DensestCore densest_level(const unsigned long long *hv, const unsigned long long *he, uint32_t n_bins, uint64_t n, uint64_t n_edges) {
    DensestCore best{0, n, n_edges, n ? (double)n_edges / (double)n : 0.0};
    if (!n || !n_edges) return best;
    uint64_t v = 0, e = 0;
    best.density = -1.0;
    for (int64_t k = (int64_t)n_bins - 1; k >= 0; --k) {   // suffix sums over the levels, densest first
        v += hv[k];
        e += he[k];
        if (v == 0) continue;
        const double d = (double)e / (double)v;
        // equal density: the larger block wins; an empty level leaves the block (and the reported k) as it is
        if (d > best.density || (d == best.density && v > best.n_vertices)) best = DensestCore{(int32_t)k, v, e, d};
    }
    return best;
}

}  // namespace kg

extern "C" int kombgpu_graph_densest_core(kombgpu_graph *g, int32_t *k_star, uint32_t *n_vertices, uint64_t *n_edges,
                                          double *density) {
    using namespace kg;
    if (!g) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = g->ctx;
    if (!g->has_core) return ctx_fail(ctx, KOMBGPU_ESTATE, "kombgpu_graph_densest_core needs kombgpu_coreness first");
    if (g->n_edges && !g->edges) return ctx_fail(ctx, KOMBGPU_ESTATE, "graph was adopted from a CSR: no canonical edge list");
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    const uint32_t n_bins = g->n && g->n_edges ? (uint32_t)g->st.max_coreness + 1 : 0u;
    std::vector<unsigned long long> h(2 * (size_t)n_bins);
    if (n_bins) {
        DevBuf<unsigned long long> hist;
        KG_ALLOC(ctx, hist, 2 * (size_t)n_bins);
        KG_CUDA(ctx, cudaMemsetAsync(hist.p, 0, 2 * (size_t)n_bins * sizeof(unsigned long long), ctx->stream));
        KG_TRY(level_histogram(ctx, g->core, nullptr, g->n, n_bins, hist.p));
        KG_TRY(level_histogram(ctx, g->core, g->edges, g->n_edges, n_bins, hist.p + n_bins));
        KG_TRY(read_back(ctx, hist.p, h.data(), h.size()));
    }
    const DensestCore best = densest_level(h.data(), h.data() + n_bins, n_bins, g->n, g->n_edges);
    if (k_star) *k_star = best.k;
    if (n_vertices) *n_vertices = (uint32_t)best.n_vertices;
    if (n_edges) *n_edges = best.n_edges;
    if (density) *density = best.density;
    return KOMBGPU_OK;
}

extern "C" int kombgpu_graph_densest_block(kombgpu_graph *g, const double *weight, int use_scores, double eps, uint32_t *n_vertices,
                                           uint64_t *n_edges, double *weight_sum, double *density, uint32_t *n_passes, uint8_t *member) {
    using namespace kg;
    if (!g) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = g->ctx;
    if (!(eps >= 0.0) || eps > 1e6) return ctx_fail(ctx, KOMBGPU_EINVAL, "eps must be in [0, 1e6]");
    if (weight && use_scores) return ctx_fail(ctx, KOMBGPU_EINVAL, "give weights or ask for the CORE-A scores, not both");
    if (use_scores && !g->has_score) return ctx_fail(ctx, KOMBGPU_ESTATE, "the CORE-A scores have not been computed");
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    const uint32_t n = g->n;
    const uint64_t launches0 = ctx->launches;
    DevBuf<double> w_dev;
    const double *w = use_scores ? g->score : nullptr;
    double W = 0.0;
    if (weight && n) {
        KG_ALLOC(ctx, w_dev, n);
        KG_CUDA(ctx, cudaMemcpyAsync(w_dev.p, weight, (size_t)n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        w = w_dev.p;
        for (uint32_t i = 0; i < n; ++i) {
            if (!(weight[i] >= 0.0) || weight[i] > 1e300) return ctx_fail(ctx, KOMBGPU_EINVAL, "weights must be finite and >= 0");
            W += weight[i];
        }
    }
    DevBuf<uint32_t> pass, list;
    DevBuf<int32_t> deg_s;
    DevBuf<BlockPass> st(ctx, 1);
    KG_ALLOC(ctx, pass, n);
    KG_ALLOC(ctx, list, n);
    KG_ALLOC(ctx, deg_s, n);
    if (!st) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
    KG_CUDA(ctx, cudaMemsetAsync(pass.p, 0xff, (size_t)(n ? n : 1) * sizeof(uint32_t), ctx->stream));
    if (n) KG_CUDA(ctx, cudaMemcpyAsync(deg_s.p, g->deg, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToDevice, ctx->stream));
    if (use_scores) KG_TRY(block_weight_sum(ctx, w, deg_s.p, n, list.p, st.p, &W));
    GraphBlockSteps steps(ctx, g, w, deg_s.p, pass.p, list.p, st.p);
    DensestBlock best{};
    KG_TRY(densest_block_passes(ctx, n, g->n_edges, W, eps, steps, &best));
    KG_TRY(block_member(ctx, pass.p, n, best.t_best, member));
    g->st.kernel_launches += ctx->launches - launches0;
    if (n_vertices) *n_vertices = (uint32_t)best.n_vertices;
    if (n_edges) *n_edges = best.n_edges;
    if (weight_sum) *weight_sum = best.weight_sum;
    if (density) *density = best.density;
    if (n_passes) *n_passes = best.passes;
    return KOMBGPU_OK;
}
