// truss.cu — the consumers of the coreness the reference keeps behind `runCore` (SURVEY.md section 8(f), row N3):
// the induced subgraph of the maximal core and the trussness of its edges.
//
// Restates Kgraph::runTruss (src/graph.cpp:486-563; disabled at :478 in the reference's main path):
//   subgraph_nodes = { v : coreness(v) == max coreness }        src/graph.cpp:470-476 (collected by runCore)
//   igraph_induced_subgraph_map                                 :502   -> flag / scan / compact, ids relabelled in order
//   igraph_trussness                                            :508   -> support counting + frontier peel over EDGES
//   nodes of the edges whose trussness is the maximum           :519-533
// trussness(e) = the largest k such that e lies in a k-truss (every edge of a k-truss closes >= k - 2 triangles
// inside it); edges in no triangle have trussness 2.  It is a unique function of the graph, so any correct
// implementation is an exact oracle (checked against networkx.k_truss and a Python restatement in tests/).
//
// Device side: the peel machinery of the k-core, on edges.  Level s = k - 2: the frontier holds the alive edges whose
// support is <= s; removing an edge destroys its triangles, which costs the other two edges of each one support;
// an edge whose support reaches s joins the next frontier.  Every row of the sub-CSR is sorted, so triangles are
// found by merging two rows, and `eid` maps a CSR entry to the id of its edge.
#include <vector>

#include "graph.cuh"
#include "primitives.cuh"

namespace kg {
namespace {

constexpr int kThreads = 256;

inline uint32_t grid_for(uint64_t n, int per_block, uint32_t cap) {
    uint32_t g = ceil_div_u64(n ? n : 1, per_block);
    return g < cap ? g : cap;
}

struct CoreFlagIn {
    const int32_t *core;
    int32_t kmax;
    __device__ uint32_t operator()(uint64_t v) const { return core[v] == kmax ? 1u : 0u; }
};
struct CoreFlagOut {
    uint32_t *sub_id;    // [n] compact id or ~0
    uint32_t *core_vid;  // [n_core] original id
    __device__ void operator()(uint64_t v, uint32_t pos, uint32_t flag) const {
        sub_id[v] = flag ? pos : 0xffffffffu;
        if (flag) core_vid[pos] = (uint32_t)v;
    }
};
struct SubEdgeFlagIn {
    const uint64_t *edges;
    const uint32_t *sub_id;
    __device__ uint32_t operator()(uint64_t i) const {
        const uint64_t e = edges[i];
        return (sub_id[(uint32_t)(e >> 32)] != 0xffffffffu && sub_id[(uint32_t)e] != 0xffffffffu) ? 1u : 0u;
    }
};
struct SubEdgeOut {
    const uint64_t *edges;
    const uint32_t *sub_id;
    uint64_t *out;   // relabelled: the map is monotone, so the list stays sorted and canonical
    __device__ void operator()(uint64_t i, uint32_t pos, uint32_t flag) const {
        if (!flag) return;
        const uint64_t e = edges[i];
        out[pos] = ((uint64_t)sub_id[(uint32_t)(e >> 32)] << 32) | sub_id[(uint32_t)e];
    }
};

// eid[p] = id (position in the canonical edge list) of the edge behind CSR entry p
__global__ void __launch_bounds__(kThreads) edge_ids_kernel(uint32_t n, const uint64_t *__restrict__ row_ptr, const uint32_t *__restrict__ col,
                                                            const uint32_t *__restrict__ fwd_start, uint32_t *__restrict__ eid) {
    for (uint64_t a = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; a < n; a += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t r0 = row_ptr[a], r1 = row_ptr[a + 1];
        const uint32_t nfwd = fwd_start[a + 1] - fwd_start[a];
        const uint64_t f0 = r1 - nfwd;   // row = [back | forward]
        for (uint64_t p = r0; p < r1; ++p) {
            if (p >= f0) {
                eid[p] = fwd_start[a] + (uint32_t)(p - f0);
            } else {
                const uint32_t w = col[p];   // w < a: the edge is (w, a), in w's forward part
                const uint32_t wn = fwd_start[w + 1] - fwd_start[w];
                const uint64_t wf0 = row_ptr[w + 1] - wn;
                uint32_t lo = 0, hi = wn;
                while (lo < hi) {
                    const uint32_t mid = (lo + hi) >> 1;
                    if (col[wf0 + mid] < (uint32_t)a) lo = mid + 1; else hi = mid;
                }
                eid[p] = fwd_start[w] + lo;
            }
        }
    }
}

// support[e] = triangles through edge e = |N(a) ∩ N(b)| (merge of two sorted rows)
__global__ void __launch_bounds__(kThreads) support_kernel(const uint64_t *__restrict__ edges, uint64_t m, const uint64_t *__restrict__ row_ptr,
                                                           const uint32_t *__restrict__ col, int32_t *__restrict__ sup) {
    for (uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; e < m; e += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t a = (uint32_t)(edges[e] >> 32), b = (uint32_t)edges[e];
        uint64_t i = row_ptr[a], j = row_ptr[b];
        const uint64_t ie = row_ptr[a + 1], je = row_ptr[b + 1];
        int32_t c = 0;
        while (i < ie && j < je) {
            const uint32_t x = col[i], y = col[j];
            c += x == y;
            i += x <= y;
            j += y <= x;
        }
        sup[e] = c;
    }
}

// level start: edges alive (state 0) with support <= s enter the frontier (state 1); also the smallest support above s
__global__ void __launch_bounds__(kThreads) truss_scan_kernel(const int32_t *__restrict__ sup, uint8_t *__restrict__ state, uint64_t m, int32_t s,
                                                              uint32_t *__restrict__ frontier, uint32_t *__restrict__ counters /* [0] count, [1] min */) {
    int32_t local_min = INT32_MAX;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t base = (uint64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31u); base < m; base += stride) {
        const uint64_t e = base + lane_id();
        bool take = false;
        if (e < m && state[e] == 0) {
            const int32_t v = sup[e];
            if (v <= s) take = true; else local_min = min(local_min, v);
        }
        const uint32_t tm = __ballot_sync(kFullMask, take);   // one atomic per warp
        if (tm) {
            uint32_t pos = 0;
            if (lane_id() == 0) pos = atomicAdd(&counters[0], (uint32_t)__popc(tm));
            pos = __shfl_sync(kFullMask, pos, 0) + __popc(tm & lanemask_lt());
            if (take) { state[e] = 1; frontier[pos] = (uint32_t)e; }
        }
    }
    local_min = warp_reduce_min(local_min);
    if (lane_id() == 0 && local_min != INT32_MAX) atomicMin(reinterpret_cast<int32_t *>(&counters[1]), local_min);
}

// One sub-round: every frontier edge is removed.  A triangle (e, e1, e2) dies with it; its other edges lose one
// support each -- once per triangle: when e1 is in the frontier too, only the smaller id of (e, e1) charges e2, and
// when both are, nobody is charged.  An edge whose support drops to s joins the next frontier (state 3 until the
// frontier edges have been retired, then 1).
__global__ void __launch_bounds__(kThreads) truss_process_kernel(const uint32_t *__restrict__ frontier, uint32_t n_front, const uint64_t *__restrict__ edges,
                                                                 const uint64_t *__restrict__ row_ptr, const uint32_t *__restrict__ col,
                                                                 const uint32_t *__restrict__ eid, int32_t *sup, uint8_t *state, int32_t s,
                                                                 uint32_t *__restrict__ next, uint32_t *__restrict__ n_next) {
    for (uint64_t f = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; f < n_front; f += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t e = frontier[f];
        const uint32_t a = (uint32_t)(edges[e] >> 32), b = (uint32_t)edges[e];
        uint64_t i = row_ptr[a], j = row_ptr[b];
        const uint64_t ie = row_ptr[a + 1], je = row_ptr[b + 1];
        while (i < ie && j < je) {
            const uint32_t x = col[i], y = col[j];
            if (x == y) {
                const uint32_t e1 = eid[i], e2 = eid[j];
                const uint8_t s1 = *(volatile uint8_t *)&state[e1], s2 = *(volatile uint8_t *)&state[e2];
                const bool dead1 = s1 == 2, dead2 = s2 == 2, in1 = s1 == 1, in2 = s2 == 1;
                if (!dead1 && !dead2) {   // the triangle is still there
                    uint32_t hit[2];
                    int nh = 0;
                    if (!in1 && !in2) { hit[nh++] = e1; hit[nh++] = e2; }
                    else if (in1 && !in2) { if (e < e1) hit[nh++] = e2; }
                    else if (!in1 && in2) { if (e < e2) hit[nh++] = e1; }
                    for (int h = 0; h < nh; ++h) {
                        const int32_t old = atomicSub(&sup[hit[h]], 1);
                        if (old == s + 1) {   // just reached the level: exactly one thread sees this
                            state[hit[h]] = 3;
                            next[atomicAdd(n_next, 1u)] = hit[h];
                        }
                    }
                }
            }
            i += x <= y;
            j += y <= x;
        }
    }
}

// retire the processed frontier (trussness = s + 2), arm the next one
__global__ void __launch_bounds__(kThreads) truss_retire_kernel(const uint32_t *__restrict__ frontier, uint32_t n_front, const uint32_t *__restrict__ next,
                                                                uint32_t n_next, uint8_t *__restrict__ state, int32_t *__restrict__ truss, int32_t s) {
    const uint64_t total = (uint64_t)n_front + n_next;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (uint64_t)gridDim.x * blockDim.x) {
        if (i < n_front) {
            state[frontier[i]] = 2;
            truss[frontier[i]] = s + 2;
        } else {
            state[next[i - n_front]] = 1;
        }
    }
}

struct TrussVertexMark {
    const uint64_t *edges;
    const int32_t *truss;
    int32_t tmax;
    uint32_t *flag;
};
__global__ void __launch_bounds__(kThreads) mark_truss_vertices_kernel(const uint64_t *__restrict__ edges, const int32_t *__restrict__ truss, uint64_t m,
                                                                       int32_t tmax, uint32_t *__restrict__ flag) {
    for (uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; e < m; e += (uint64_t)gridDim.x * blockDim.x)
        if (truss[e] >= tmax) {
            flag[(uint32_t)(edges[e] >> 32)] = 1u;
            flag[(uint32_t)edges[e]] = 1u;
        }
}
struct FlagIn {
    const uint32_t *flag;
    __device__ uint32_t operator()(uint64_t i) const { return flag[i]; }
};
struct TrussVidOut {
    const uint32_t *core_vid;
    uint32_t *out;
    __device__ void operator()(uint64_t i, uint32_t pos, uint32_t f) const {
        if (f) out[pos] = core_vid[i];
    }
};

__global__ void __launch_bounds__(kThreads) sub_edges_original_kernel(const uint64_t *__restrict__ sub_edges, uint64_t m,
                                                                      const uint32_t *__restrict__ core_vid, uint32_t *__restrict__ u,
                                                                      uint32_t *__restrict__ v) {
    for (uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; e < m; e += (uint64_t)gridDim.x * blockDim.x) {
        u[e] = core_vid[(uint32_t)(sub_edges[e] >> 32)];
        v[e] = core_vid[(uint32_t)sub_edges[e]];
    }
}

}  // namespace

void truss_free(kombgpu_ctx *ctx, MaxCoreTruss *tr) {
    void *ptrs[] = {tr->core_vid, tr->edges, tr->truss, tr->vertices};
    for (void *p : ptrs)
        if (p) ws_free(ctx, p);
    *tr = MaxCoreTruss{};
}

void truss_release(kombgpu_graph *g) {
    truss_free(g->ctx, &g->tr);
    g->has_truss = false;
}

int max_core_vertices(kombgpu_ctx *ctx, const int32_t *core, uint32_t n, int32_t kmax, DevBuf<uint32_t> &sub_id,
                      DevBuf<uint32_t> &core_vid, uint32_t *n_core) {
    DevBuf<uint32_t> d_cnt(ctx, 1);
    KG_ALLOC(ctx, sub_id, n);
    KG_ALLOC(ctx, core_vid, n);
    if (!d_cnt) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
    KG_TRY((device_scan<uint32_t>(ctx, n, CoreFlagIn{core, kmax}, CoreFlagOut{sub_id.p, core_vid.p}, d_cnt.p)));
    return read_back(ctx, d_cnt.p, n_core, 1);
}

int max_core_edges(kombgpu_ctx *ctx, const uint64_t *edges, uint64_t count, const uint32_t *sub_id, DevBuf<uint64_t> &out,
                   uint64_t *m) {
    DevBuf<uint32_t> d_cnt(ctx, 1);
    KG_ALLOC(ctx, out, count);
    if (!d_cnt) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
    KG_TRY((device_scan<uint32_t>(ctx, count, SubEdgeFlagIn{edges, sub_id}, SubEdgeOut{edges, sub_id, out.p}, d_cnt.p)));
    uint32_t m32 = 0;
    KG_TRY(read_back(ctx, d_cnt.p, &m32, 1));
    *m = m32;
    return KOMBGPU_OK;
}

int sub_edges_truss(kombgpu_ctx *ctx, DevBuf<uint64_t> &sub_edges, uint64_t m, DevBuf<uint32_t> &core_vid, uint32_t n_core,
                    MaxCoreTruss *tr) {
    const uint32_t cap = (uint32_t)ctx->sm_count * 8u;
    DevBuf<uint32_t> d_cnt(ctx, 2);
    if (!d_cnt) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");

    // 3. its CSR (rows sorted) and the entry -> edge id map
    kombgpu_graph sub;
    sub.ctx = ctx;
    DevBuf<uint64_t> edges_copy;   // csr_from_edges takes ownership of the list it indexes
    KG_ALLOC(ctx, edges_copy, m);
    if (m) KG_CUDA(ctx, cudaMemcpyAsync(edges_copy.p, sub_edges.p, m * sizeof(uint64_t), cudaMemcpyDeviceToDevice, ctx->stream));
    int rc = csr_from_edges(ctx, edges_copy, m, n_core, &sub);
    if (rc != KOMBGPU_OK) { graph_release(&sub); return rc; }
    DevBuf<uint32_t> eid, front_a, front_b;
    DevBuf<int32_t> sup, truss;
    DevBuf<uint8_t> state;
    auto bail = [&](int code) { graph_release(&sub); return code; };
    if (!eid.alloc(ctx, 2 * m) || !sup.alloc(ctx, m) || !truss.alloc(ctx, m) || !state.alloc(ctx, m) || !front_a.alloc(ctx, m) || !front_b.alloc(ctx, m))
        return bail(ctx_fail(ctx, KOMBGPU_ENOMEM, "truss workspace"));
    int32_t tmax = m ? 2 : 0;
    if (m) {
        edge_ids_kernel<<<grid_for(n_core, kThreads, cap), kThreads, 0, ctx->stream>>>(n_core, sub.row_ptr, sub.col, sub.fwd_start, eid.p);
        support_kernel<<<grid_for(m, kThreads, cap), kThreads, 0, ctx->stream>>>(sub.edges, m, sub.row_ptr, sub.col, sup.p);
        ctx->launches += 2;
        cudaMemsetAsync(state.p, 0, m, ctx->stream);
        // 4. peel the edges level by level
        uint64_t alive = m;
        int32_t s = 0;
        uint32_t *fa = front_a.p, *fb = front_b.p;
        while (alive) {
            const uint32_t init[2] = {0u, (uint32_t)INT32_MAX};
            cudaMemcpyAsync(d_cnt.p, init, sizeof(init), cudaMemcpyHostToDevice, ctx->stream);
            truss_scan_kernel<<<grid_for(m, kThreads, cap), kThreads, 0, ctx->stream>>>(sup.p, state.p, m, s, fa, d_cnt.p);
            ctx->launches++;
            uint32_t h[2] = {0, 0};
            rc = read_back(ctx, d_cnt.p, h, 2);
            if (rc != KOMBGPU_OK) return bail(rc);
            uint32_t n_front = h[0];
            if (n_front == 0) {   // empty level: jump to the smallest support left
                if (h[1] == (uint32_t)INT32_MAX) return bail(ctx_fail(ctx, KOMBGPU_EINTERNAL, "truss peel lost %llu edges", (unsigned long long)alive));
                s = (int32_t)h[1];
                continue;
            }
            tmax = s + 2;
            while (n_front) {
                cudaMemsetAsync(d_cnt.p, 0, sizeof(uint32_t), ctx->stream);
                truss_process_kernel<<<grid_for(n_front, 64, cap * 4), 64, 0, ctx->stream>>>(fa, n_front, sub.edges, sub.row_ptr, sub.col, eid.p, sup.p,
                                                                                             state.p, s, fb, d_cnt.p);
                ctx->launches++;
                uint32_t n_next = 0;
                rc = read_back(ctx, d_cnt.p, &n_next, 1);
                if (rc != KOMBGPU_OK) return bail(rc);
                truss_retire_kernel<<<grid_for((uint64_t)n_front + n_next, kThreads, cap), kThreads, 0, ctx->stream>>>(fa, n_front, fb, n_next, state.p,
                                                                                                                      truss.p, s);
                ctx->launches++;
                alive -= n_front;
                n_front = n_next;
                uint32_t *t = fa; fa = fb; fb = t;
            }
            s += 1;
        }
    }
    cudaError_t ke = cudaPeekAtLastError();
    if (ke != cudaSuccess) return bail(ctx_fail(ctx, KOMBGPU_ECUDA, "truss kernels: %s", cudaGetErrorString(ke)));

    // 5. the unitigs of the edges of maximal trussness (src/graph.cpp:519-533)
    DevBuf<uint32_t> vflag, tverts;
    if (!vflag.alloc(ctx, n_core) || !tverts.alloc(ctx, n_core)) return bail(ctx_fail(ctx, KOMBGPU_ENOMEM, "truss workspace"));
    cudaMemsetAsync(vflag.p, 0, (size_t)(n_core ? n_core : 1) * sizeof(uint32_t), ctx->stream);
    if (m) {
        mark_truss_vertices_kernel<<<grid_for(m, kThreads, cap), kThreads, 0, ctx->stream>>>(sub.edges, truss.p, m, tmax, vflag.p);
        ctx->launches++;
    }
    rc = device_scan<uint32_t>(ctx, n_core, FlagIn{vflag.p}, TrussVidOut{core_vid.p, tverts.p}, d_cnt.p);
    if (rc != KOMBGPU_OK) return bail(rc);
    uint32_t n_tv = 0;
    rc = read_back(ctx, d_cnt.p, &n_tv, 1);
    if (rc != KOMBGPU_OK) return bail(rc);
    graph_release(&sub);
    tr->n_core = n_core;
    tr->m = m;
    tr->tmax = tmax;
    tr->n_vertices = n_tv;
    tr->core_vid = core_vid.take();
    tr->edges = sub_edges.take();
    tr->truss = truss.take();
    tr->vertices = tverts.take();
    return KOMBGPU_OK;
}

int max_core_truss(kombgpu_graph *g) {
    kombgpu_ctx *ctx = g->ctx;
    truss_release(g);
    // 1. the vertices of the maximal core, relabelled in order
    DevBuf<uint32_t> sub_id, core_vid;
    uint32_t n_core = 0;
    KG_TRY(max_core_vertices(ctx, g->core, g->n, g->st.max_coreness, sub_id, core_vid, &n_core));
    // 2. the induced edges
    DevBuf<uint64_t> sub_edges;
    uint64_t m = 0;
    KG_TRY(max_core_edges(ctx, g->edges, g->n_edges, sub_id.p, sub_edges, &m));
    sub_id.release();
    // 3-5. their trussness
    KG_TRY(sub_edges_truss(ctx, sub_edges, m, core_vid, n_core, &g->tr));
    g->has_truss = true;
    return KOMBGPU_OK;
}

int truss_edges_to_host(kombgpu_ctx *ctx, const MaxCoreTruss &tr, uint32_t *u, uint32_t *v, int32_t *trussness) {
    const uint64_t m = tr.m;
    if (m == 0) return KOMBGPU_OK;
    if (u || v) {
        if (!u || !v) return ctx_fail(ctx, KOMBGPU_EINVAL, "u and v must be given together");
        DevBuf<uint32_t> du, dv;
        KG_ALLOC(ctx, du, m);
        KG_ALLOC(ctx, dv, m);
        KG_LAUNCH(ctx, sub_edges_original_kernel, grid_for(m, kThreads, (uint32_t)ctx->sm_count * 8u), kThreads, 0, tr.edges, m, tr.core_vid, du.p, dv.p);
        KG_CUDA(ctx, cudaMemcpyAsync(u, du.p, m * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
        KG_CUDA(ctx, cudaMemcpyAsync(v, dv.p, m * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
        KG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    if (trussness) {
        KG_CUDA(ctx, cudaMemcpyAsync(trussness, tr.truss, m * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
        KG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return KOMBGPU_OK;
}

int truss_vertices_to_host(kombgpu_ctx *ctx, const MaxCoreTruss &tr, uint32_t *vids) {
    if (tr.n_vertices == 0) return KOMBGPU_OK;
    if (!vids) return ctx_fail(ctx, KOMBGPU_EINVAL, "null argument");
    KG_CUDA(ctx, cudaMemcpyAsync(vids, tr.vertices, (size_t)tr.n_vertices * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    KG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return KOMBGPU_OK;
}

}  // namespace kg

using namespace kg;

extern "C" {

int kombgpu_graph_max_core_truss(kombgpu_graph *g, uint32_t *n_core_vertices, uint64_t *n_core_edges, int32_t *max_trussness,
                                 uint32_t *n_truss_vertices) {
    if (!g) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = g->ctx;
    if (!g->has_core) return ctx_fail(ctx, KOMBGPU_ESTATE, "kombgpu_graph_max_core_truss needs kombgpu_coreness first");
    if (g->n_edges && !g->edges) return ctx_fail(ctx, KOMBGPU_ESTATE, "graph was adopted from a CSR: no canonical edge list");
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    if (!g->has_truss) KG_TRY(max_core_truss(g));
    if (n_core_vertices) *n_core_vertices = g->tr.n_core;
    if (n_core_edges) *n_core_edges = g->tr.m;
    if (max_trussness) *max_trussness = g->tr.tmax;
    if (n_truss_vertices) *n_truss_vertices = g->tr.n_vertices;
    return KOMBGPU_OK;
}

int kombgpu_graph_max_core_edges(const kombgpu_graph *g, uint32_t *u, uint32_t *v, int32_t *trussness) {
    if (!g) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = g->ctx;
    if (!g->has_truss) return ctx_fail(ctx, KOMBGPU_ESTATE, "call kombgpu_graph_max_core_truss first");
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    return truss_edges_to_host(ctx, g->tr, u, v, trussness);
}

int kombgpu_graph_truss_vertices(const kombgpu_graph *g, uint32_t *vids) {
    if (!g) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = g->ctx;
    if (!g->has_truss) return ctx_fail(ctx, KOMBGPU_ESTATE, "call kombgpu_graph_max_core_truss first");
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    return truss_vertices_to_host(ctx, g->tr, vids);
}

}  // extern "C"
