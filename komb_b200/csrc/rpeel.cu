// rpeel.cu — stage 2 over the ranks of a communicator when the WHOLE graph is small: every rank gathers the other
// ranks' rows out of peer memory and peels the whole graph with the single-GPU kernel (peel.cu), then keeps its slice.
//
// Replaces igraph_coreness (src/graph.cpp:463).  A partitioned peel pays a remote hop (asynchronous, apeel.cu) or a
// meeting of all ranks (log-based, ppeel.cu) for every one of the hundreds of dependent generations of a collapsing
// core; a graph that one GPU peels in a few milliseconds is not worth that.  Measured on cfg2 x 2 / x 4 (131 M / 263 M
// adjacency entries in all): 5.5 / 8.4 ms replicated against 9.3 / 18.6 ms asynchronous.  The build, CORE-A and every
// result stay partitioned; nothing but the adjacency crosses a link (4 bytes per entry per rank, pulled by plain
// device-to-device copies out of the symmetric heap).
#include "dgraph.cuh"

namespace kg {
namespace {

constexpr int kThreads = 256;

// rows of rank q: row_ptr_full[base + r] = off + rp[r] (r = 0 .. n_rows), deg_full[base + r] = rp[r + 1] - rp[r]
__global__ void __launch_bounds__(kThreads) place_rows_kernel(const uint32_t *__restrict__ rp, uint32_t n_rows, uint64_t off, uint64_t *__restrict__ row_ptr_full,
                                                              int32_t *__restrict__ deg_full) {
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r <= n_rows; r += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t a = rp[r];
        row_ptr_full[r] = off + a;
        if (r < n_rows) deg_full[r] = (int32_t)(rp[r + 1] - a);
    }
}

}  // namespace

int dist_peel_replicated(kombgpu_dist_graph *g, int rc) {
    kombgpu_comm *c = g->comm;
    kombgpu_ctx *ctx = g->ctx;
    const int world = c->world;
    const uint32_t n_local = g->n_local, n_global = g->n_global;
    if (!g->row_ptr32) return ctx_fail(ctx, KOMBGPU_ESTATE, "the replicated peel needs the rank's rows");

    // every rank's share of the adjacency
    unsigned long long mine = g->n_directed, all_dir[kMaxRanks];
    KG_TRY(exchange_rc(c, rc, &mine, 1, all_dir));
    uint64_t total = 0, max_dir = 0, off[kMaxRanks + 1] = {};
    for (int q = 0; q < world; ++q) {
        off[q] = total;
        total += all_dir[q];
        max_dir = all_dir[q] > max_dir ? all_dir[q] : max_dir;
    }
    off[world] = total;
    if (total >= (1ull << 32)) return ctx_fail(ctx, KOMBGPU_EINVAL, "graph too large for the replicated peel");   // on every rank

    // the rows go into the symmetric heap, where the peers can read them
    SymRewind heap{c, sym_mark(c)};
    uint32_t *col_sym = nullptr, *rp_sym = nullptr;
    PeerPtrs<uint32_t> col_peers{}, rp_peers{};
    rc = sym_alloc(c, (size_t)max_dir, &col_sym, &col_peers);
    rc = first_rc(rc, sym_alloc(c, (size_t)g->step + 1, &rp_sym, &rp_peers));
    if (rc == KOMBGPU_OK) rc = [&]() -> int {
        if (g->n_directed) KG_CUDA(ctx, cudaMemcpyAsync(col_sym, g->col, g->n_directed * sizeof(uint32_t), cudaMemcpyDeviceToDevice, ctx->stream));
        KG_CUDA(ctx, cudaMemcpyAsync(rp_sym, g->row_ptr32, ((size_t)n_local + 1) * sizeof(uint32_t), cudaMemcpyDeviceToDevice, ctx->stream));
        return KOMBGPU_OK;
    }();
    KG_TRY(barrier_rc(c, rc));   // every rank's rows are in place

    kombgpu_graph whole;
    whole.ctx = ctx;
    whole.n = n_global;
    whole.n_edges = total / 2;
    whole.st.max_coreness = -1;
    auto fail = [&](int rc) { graph_release(&whole); return rc; };
    rc = [&]() -> int {
        whole.row_ptr = static_cast<uint64_t *>(ws_alloc(ctx, ((size_t)n_global + 1) * sizeof(uint64_t)));
        whole.col = static_cast<uint32_t *>(ws_alloc(ctx, (size_t)(total ? total : 1) * sizeof(uint32_t)));
        whole.deg = static_cast<int32_t *>(ws_alloc(ctx, (size_t)(n_global ? n_global : 1) * sizeof(int32_t)));
        if (!whole.row_ptr || !whole.col || !whole.deg) return ctx_fail(ctx, KOMBGPU_ENOMEM, "the whole graph's CSR");
        for (int q = 0; q < world; ++q) {
            const uint64_t lo = (uint64_t)q * g->step;
            const uint32_t rows_q = lo < n_global ? (uint32_t)((lo + g->step < n_global ? lo + g->step : n_global) - lo) : 0u;
            if (all_dir[q]) {
                const cudaError_t e = cudaMemcpyAsync(whole.col + off[q], col_peers.p[q], all_dir[q] * sizeof(uint32_t), cudaMemcpyDeviceToDevice, ctx->stream);
                if (e != cudaSuccess) return ctx_fail(ctx, KOMBGPU_ECUDA, "copy of rank %d's rows: %s", q, cudaGetErrorString(e));
            }
            if (lo <= n_global && (rows_q || lo == n_global)) {
                place_rows_kernel<<<min(ceil_div_u64((uint64_t)rows_q + 1, kThreads), 148u * 8u), kThreads, 0, ctx->stream>>>(
                    rp_peers.p[q], rows_q, off[q], whole.row_ptr + lo, whole.deg + (lo < n_global ? lo : 0));
                ctx->launches++;
            }
        }
        const cudaError_t e = cudaPeekAtLastError();
        if (e != cudaSuccess) return ctx_fail(ctx, KOMBGPU_ECUDA, "place_rows_kernel: %s", cudaGetErrorString(e));
        return KOMBGPU_OK;
    }();
    rc = barrier_rc(c, rc);   // everybody has read everybody's rows: the symmetric buffers may go
    if (rc != KOMBGPU_OK) return fail(rc);

    rc = peel_coreness(&whole);
    if (rc != KOMBGPU_OK) return fail(rc);
    if (n_local) {
        const cudaError_t e = cudaMemcpyAsync(g->core, whole.core + g->v_lo, (size_t)n_local * sizeof(int32_t), cudaMemcpyDeviceToDevice, ctx->stream);
        if (e != cudaSuccess) return fail(ctx_fail(ctx, KOMBGPU_ECUDA, "coreness slice: %s", cudaGetErrorString(e)));
    }
    g->st.max_coreness = whole.st.max_coreness;
    g->st.peel_levels = whole.st.peel_levels;
    g->st.peel_subrounds = 0;        // the ranks never meet inside the peel
    g->st.peel_solo_subrounds = 0;
    g->st.n_messages_sent = 0;
    g->st.n_messages_recv = total - g->n_directed;   // adjacency entries pulled from the peers
    g->st.peel_async = 2;
    KG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    graph_release(&whole);
    return KOMBGPU_OK;
}

}  // namespace kg
