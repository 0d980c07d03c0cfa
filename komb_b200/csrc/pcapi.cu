// pcapi.cu — extern "C" entry points of the peer-memory multi-GPU path (include/kombgpu.h, "multi-GPU, peer-memory
// path"): one rank's handle on a graph partitioned by unitig-id range.  Every compute call is collective over the
// ranks of the communicator.
#include <new>

#include "dgraph.cuh"
#include "kombgpu_debug.h"

using namespace kg;

namespace {

__global__ void unpack_local_edges_kernel(const uint64_t *__restrict__ edges, uint64_t n, uint32_t *__restrict__ u, uint32_t *__restrict__ v) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t e = edges[i];
        if (u) u[i] = (uint32_t)(e >> 32);
        if (v) v[i] = (uint32_t)e;
    }
}

__global__ void widen_local_kernel(const uint32_t *__restrict__ in, uint64_t count, uint64_t *__restrict__ out) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (uint64_t)gridDim.x * blockDim.x) out[i] = in[i];
}

template <typename T>
int fetch(kombgpu_ctx *ctx, const T *dev, T *host, size_t count) {
    if (!host || count == 0) return KOMBGPU_OK;
    KG_CUDA(ctx, cudaMemcpyAsync(host, dev, count * sizeof(T), cudaMemcpyDeviceToHost, ctx->stream));
    KG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return KOMBGPU_OK;
}

int dist_build_common(kombgpu_comm *c, const uint32_t *a, const uint32_t *b, uint64_t count, uint32_t n_global, bool from_hits,
                      kombgpu_dist_graph **out) {
    if (!c) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = c->ctx;
    if (!out || (count && (!a || !b))) return ctx_fail(ctx, KOMBGPU_EINVAL, "null argument");
    *out = nullptr;
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    kombgpu_dist_graph *g = new (std::nothrow) kombgpu_dist_graph();
    if (!g) return ctx_fail(ctx, KOMBGPU_ENOMEM, "host allocation");
    const int rc = dist_build(c, a, b, count, n_global, from_hits, g);
    if (rc != KOMBGPU_OK) {
        dist_graph_release(g);
        delete g;
        return rc;
    }
    *out = g;
    return KOMBGPU_OK;
}

}  // namespace

extern "C" {

int kombgpu_dist_build_hits_dev(kombgpu_comm *c, const uint32_t *read_key, const uint32_t *unitig, uint64_t n_hits, uint32_t n_global,
                                kombgpu_dist_graph **out) {
    return dist_build_common(c, read_key, unitig, n_hits, n_global, true, out);
}

int kombgpu_dist_build_pairs_dev(kombgpu_comm *c, const uint32_t *u, const uint32_t *v, uint64_t n_pairs, uint32_t n_global,
                                 kombgpu_dist_graph **out) {
    return dist_build_common(c, u, v, n_pairs, n_global, false, out);
}

// host-pointer forms: the rank's share is uploaded first (what a host without CUDA headers calls, e.g. komb2)
static int dist_build_host(kombgpu_comm *c, const uint32_t *a, const uint32_t *b, uint64_t count, uint32_t n_global, bool from_hits,
                           kombgpu_dist_graph **out) {
    if (!c) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = c->ctx;
    if (!out || (count && (!a || !b))) return ctx_fail(ctx, KOMBGPU_EINVAL, "null argument");
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    DevBuf<uint32_t> da, db;
    KG_ALLOC(ctx, da, count);
    KG_ALLOC(ctx, db, count);
    if (count) {
        KG_CUDA(ctx, cudaMemcpyAsync(da.p, a, count * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
        KG_CUDA(ctx, cudaMemcpyAsync(db.p, b, count * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    }
    return dist_build_common(c, da.p, db.p, count, n_global, from_hits, out);
}

int kombgpu_dist_build_hits(kombgpu_comm *c, const uint32_t *read_key, const uint32_t *unitig, uint64_t n_hits, uint32_t n_global,
                            kombgpu_dist_graph **out) {
    return dist_build_host(c, read_key, unitig, n_hits, n_global, true, out);
}

int kombgpu_dist_build_pairs(kombgpu_comm *c, const uint32_t *u, const uint32_t *v, uint64_t n_pairs, uint32_t n_global,
                             kombgpu_dist_graph **out) {
    return dist_build_host(c, u, v, n_pairs, n_global, false, out);
}

int kombgpu_dist_coreness(kombgpu_dist_graph *g) {
    if (!g) return KOMBGPU_EINVAL;
    KG_CUDA(g->ctx, cudaSetDevice(g->ctx->device));
    if (g->has_core) return KOMBGPU_OK;
    kombgpu_ctx *ctx = g->ctx;
    EvTimer timer(ctx);
    int rc = KOMBGPU_OK;
    if (!g->core) {
        g->core = static_cast<int32_t *>(ws_alloc(ctx, (g->n_local ? g->n_local : 1) * sizeof(int32_t)));
        if (!g->core) rc = ctx_fail(ctx, KOMBGPU_ENOMEM, "coreness array");
    }
    // what the build prepared for (KOMBGPU_DIST_PEEL, or the shape of the graph)
    rc = g->peel_choice == 2 ? dist_peel_replicated(g, rc) : (g->peel_choice == 1 ? dist_peel_async(g, rc) : dist_peel(g, rc));
    if (rc != KOMBGPU_OK) return rc;
    g->st.ms_peel = timer.lap();
    g->has_core = true;
    return KOMBGPU_OK;
}

int kombgpu_dist_corea(kombgpu_dist_graph *g, int key_mode) {
    if (!g) return KOMBGPU_EINVAL;
    if (!g->has_core) return ctx_fail(g->ctx, KOMBGPU_ESTATE, "kombgpu_dist_corea needs kombgpu_dist_coreness first");
    KG_CUDA(g->ctx, cudaSetDevice(g->ctx->device));
    return dist_corea(g, key_mode);
}

void kombgpu_dist_graph_destroy(kombgpu_dist_graph *g) {
    if (!g) return;
    dist_graph_release(g);
    delete g;
}

int kombgpu_dist_graph_stats(const kombgpu_dist_graph *g, kombgpu_dist_stats *out) {
    if (!g || !out) return KOMBGPU_EINVAL;
    *out = g->st;
    return KOMBGPU_OK;
}

int kombgpu_dist_graph_results(const kombgpu_dist_graph *g, int32_t *degree, int32_t *coreness, double *score) {
    if (!g) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = g->ctx;
    if (coreness && !g->has_core) return ctx_fail(ctx, KOMBGPU_ESTATE, "coreness not computed yet");
    if (score && !g->has_score) return ctx_fail(ctx, KOMBGPU_ESTATE, "CORE-A not computed yet");
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    KG_TRY(fetch(ctx, g->deg, degree, g->n_local));
    KG_TRY(fetch(ctx, g->core, coreness, g->n_local));
    return fetch(ctx, g->score, score, g->n_local);
}

int kombgpu_dist_graph_edges(const kombgpu_dist_graph *g, uint32_t *u, uint32_t *v, uint32_t *mult) {
    if (!g) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = g->ctx;
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    const uint64_t m = g->n_fwd;
    if (m && (u || v)) {
        DevBuf<uint32_t> du, dv;
        if (u) KG_ALLOC(ctx, du, m);
        if (v) KG_ALLOC(ctx, dv, m);
        KG_LAUNCH(ctx, unpack_local_edges_kernel, min(ceil_div_u64(m, 256), (uint32_t)ctx->sm_count * 8u), 256, 0, g->edges, m, du.p, dv.p);
        KG_TRY(fetch(ctx, du.p, u, m));
        KG_TRY(fetch(ctx, dv.p, v, m));
    }
    return fetch(ctx, g->mult, mult, m);
}

int kombgpu_dist_graph_edges_csr(const kombgpu_dist_graph *g, uint64_t *fwd_ptr, uint32_t *v) {
    if (!g) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = g->ctx;
    if (!fwd_ptr || (g->n_fwd && !v)) return ctx_fail(ctx, KOMBGPU_EINVAL, "null argument");
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    const uint64_t m = g->n_fwd;
    DevBuf<uint32_t> dv;
    DevBuf<uint64_t> dp;
    KG_ALLOC(ctx, dp, (size_t)g->n_local + 1);
    KG_LAUNCH(ctx, widen_local_kernel, min(ceil_div_u64((uint64_t)g->n_local + 1, 256), (uint32_t)ctx->sm_count * 8u), 256, 0, g->fwd_start,
              (uint64_t)g->n_local + 1, dp.p);
    if (m) {
        KG_ALLOC(ctx, dv, m);
        KG_LAUNCH(ctx, unpack_local_edges_kernel, min(ceil_div_u64(m, 256), (uint32_t)ctx->sm_count * 8u), 256, 0, g->edges, m,
                  (uint32_t *)nullptr, dv.p);
    }
    KG_TRY(fetch(ctx, dp.p, fwd_ptr, (size_t)g->n_local + 1));
    return fetch(ctx, dv.p, v, m);
}

int kombgpu_dist_graph_device_arrays(const kombgpu_dist_graph *g, const uint64_t **row_ptr, const uint32_t **col,
                                     const uint64_t **edges_packed, const int32_t **degree, const int32_t **coreness,
                                     const double **score) {
    if (!g) return KOMBGPU_EINVAL;
    if (row_ptr) *row_ptr = nullptr;   // the partitioned path keeps its adjacency grouped by neighbour (dgraph.cuh), not as rows
    if (col) *col = nullptr;
    if (edges_packed) *edges_packed = g->edges;
    if (degree) *degree = g->deg;
    if (coreness) *coreness = g->has_core ? g->core : nullptr;
    if (score) *score = g->has_score ? g->score : nullptr;
    return KOMBGPU_OK;
}

// measurement aid (include/kombgpu_debug.h): how many rounds the build reduced its pairs in
int kombgpu_debug_dist_build_rounds(const kombgpu_dist_graph *g, uint32_t *n_rounds) {
    if (!g || !n_rounds) return KOMBGPU_EINVAL;
    *n_rounds = g->build_rounds;
    return KOMBGPU_OK;
}

int kombgpu_dist_graph_summary(const kombgpu_dist_graph *g, int32_t *max_coreness, double *max_score) {
    if (!g) return KOMBGPU_EINVAL;
    if (!g->has_core) return ctx_fail(g->ctx, KOMBGPU_ESTATE, "coreness not computed yet");
    if (max_coreness) *max_coreness = g->st.max_coreness;
    if (max_score) *max_score = g->has_score ? g->max_score : 0.0;
    return KOMBGPU_OK;
}

}  // extern "C"
