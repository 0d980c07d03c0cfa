// capi.cu — the extern "C" boundary of libkombgpu.so (include/kombgpu.h):
// context + workspace arena, host<->device staging, stage sequencing and timing.
#include <cstdarg>
#include <cstring>
#include <new>

#include "graph.cuh"
#include "kombgpu_debug.h"

namespace kg {
namespace { __global__ void small_copy_kernel(const unsigned char *__restrict__ src, unsigned char *dst, uint32_t bytes); }

int small_read_back(kombgpu_ctx *ctx, const void *dev, void *host, size_t bytes) {
    small_copy_kernel<<<1, 256, 0, ctx->stream>>>(static_cast<const unsigned char *>(dev), static_cast<unsigned char *>(ctx->pinned),
                                                  (uint32_t)bytes);
    ctx->launches++;
    KG_CUDA(ctx, cudaPeekAtLastError());
    KG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    memcpy(host, ctx->pinned, bytes);
    return KOMBGPU_OK;
}

static thread_local std::string g_create_error;

int ctx_fail(kombgpu_ctx *ctx, int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (ctx) ctx->err = buf; else g_create_error = buf;
    if (code == KOMBGPU_ECUDA) cudaGetLastError();  // clear the sticky-free error state
    return code;
}

// ---- workspace arena ---------------------------------------------------------
// Device memory is cached per context: a steady-state run of the path performs
// no cudaMalloc/cudaFree at all.
void *ws_alloc(kombgpu_ctx *ctx, size_t bytes) {
    bytes = (bytes + 511) & ~(size_t)511;
    if (bytes == 0) bytes = 512;
    int best = -1;
    for (size_t i = 0; i < ctx->arena.size(); ++i) {
        const ArenaBlock &b = ctx->arena[i];
        if (b.in_use || b.bytes < bytes) continue;
        if (b.bytes > 2 * bytes + (1u << 20)) continue;  // do not burn a huge block on a tiny request
        if (best < 0 || b.bytes < ctx->arena[best].bytes) best = (int)i;
    }
    if (best >= 0) {
        ctx->arena[best].in_use = true;
        return ctx->arena[best].ptr;
    }
    void *p = nullptr;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e != cudaSuccess) {
        cudaGetLastError();
        // give cached-but-idle blocks back and retry once
        cudaStreamSynchronize(ctx->stream);
        for (size_t i = 0; i < ctx->arena.size();) {
            if (!ctx->arena[i].in_use) {
                cudaFree(ctx->arena[i].ptr);
                ctx->arena.erase(ctx->arena.begin() + i);
            } else {
                ++i;
            }
        }
        e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess) { cudaGetLastError(); return nullptr; }
    }
    ctx->arena.push_back(ArenaBlock{p, bytes, true});
    return p;
}

void ws_free(kombgpu_ctx *ctx, void *p) {
    if (!p) return;
    for (auto &b : ctx->arena)
        if (b.ptr == p) { b.in_use = false; return; }
}

void ws_release(kombgpu_ctx *ctx, void *p) {
    if (!p) return;
    for (size_t i = 0; i < ctx->arena.size(); ++i)
        if (ctx->arena[i].ptr == p) {
            cudaStreamSynchronize(ctx->stream);
            cudaFree(p);
            ctx->arena.erase(ctx->arena.begin() + i);
            return;
        }
}

void ws_trim(kombgpu_ctx *ctx) {
    cudaStreamSynchronize(ctx->stream);
    for (size_t i = 0; i < ctx->arena.size();) {
        if (!ctx->arena[i].in_use) {
            cudaFree(ctx->arena[i].ptr);
            ctx->arena.erase(ctx->arena.begin() + i);
        } else {
            ++i;
        }
    }
}

namespace {

// stage timing with the context's own event pair (stages never nest)
struct StageTimer {
    kombgpu_ctx *ctx;
    explicit StageTimer(kombgpu_ctx *c) : ctx(c) { cudaEventRecord(ctx->ev_a, ctx->stream); }
    float stop() {
        float ms = 0.f;
        cudaEventRecord(ctx->ev_b, ctx->stream);
        cudaEventSynchronize(ctx->ev_b);
        cudaEventElapsedTime(&ms, ctx->ev_a, ctx->ev_b);
        return ms;
    }
};

template <typename T>
int upload(kombgpu_ctx *ctx, DevBuf<T> &dst, const T *host, size_t count) {
    KG_ALLOC(ctx, dst, count);
    if (count) KG_CUDA(ctx, cudaMemcpyAsync(dst.p, host, count * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
    return KOMBGPU_OK;
}

template <typename T>
int download(kombgpu_ctx *ctx, const T *dev, T *host, size_t count) {
    if (count == 0) return KOMBGPU_OK;
    KG_CUDA(ctx, cudaMemcpyAsync(host, dev, count * sizeof(T), cudaMemcpyDeviceToHost, ctx->stream));
    KG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return KOMBGPU_OK;
}

__global__ void small_copy_kernel(const unsigned char *__restrict__ src, unsigned char *dst, uint32_t bytes) {
    for (uint32_t i = threadIdx.x; i < bytes; i += blockDim.x) dst[i] = src[i];
}

__global__ void unpack_edges_kernel(const uint64_t *__restrict__ edges, uint64_t n_edges, uint32_t *__restrict__ u,
                                    uint32_t *__restrict__ v) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_edges; i += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t e = edges[i];
        u[i] = (uint32_t)(e >> 32);
        v[i] = (uint32_t)e;
    }
}

// CSR form of the edge list: the targets alone (the sources are implied by the forward index)
__global__ void edge_targets_kernel(const uint64_t *__restrict__ edges, uint64_t n_edges, uint32_t *__restrict__ v) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_edges; i += (uint64_t)gridDim.x * blockDim.x)
        v[i] = (uint32_t)edges[i];
}
__global__ void widen_u32_kernel(const uint32_t *__restrict__ in, uint64_t count, uint64_t *__restrict__ out) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (uint64_t)gridDim.x * blockDim.x) out[i] = in[i];
}

// Start the download of the canonical edge list on the copy stream, behind everything queued on the compute stream so
// far.  Pair form: u[E], v[E]; CSR form (fwd_ptr != nullptr): fwd_ptr[n + 1], v[E] -- half the bytes.
// The staging buffers must stay alive until the copy stream has drained.
struct EdgeDownload {
    DevBuf<uint32_t> du, dv;
    DevBuf<uint64_t> dptr;
    bool in_flight = false;
};
int start_edge_download(kombgpu_ctx *ctx, const kombgpu_graph *g, const uint64_t *edges, uint64_t E, uint32_t n, uint32_t *u,
                        uint64_t *fwd_ptr, uint32_t *v, EdgeDownload &dl) {
    const uint32_t grid = min(ceil_div_u64(E ? E : 1, 256), (uint32_t)ctx->sm_count * 8u);
    if (E) {
        KG_ALLOC(ctx, dl.dv, E);
        if (fwd_ptr) {
            KG_LAUNCH(ctx, edge_targets_kernel, grid, 256, 0, edges, E, dl.dv.p);
        } else {
            KG_ALLOC(ctx, dl.du, E);
            KG_LAUNCH(ctx, unpack_edges_kernel, grid, 256, 0, edges, E, dl.du.p, dl.dv.p);
        }
    }
    if (fwd_ptr) {
        KG_ALLOC(ctx, dl.dptr, (size_t)n + 1);
        KG_LAUNCH(ctx, widen_u32_kernel, min(ceil_div_u64((uint64_t)n + 1, 256), (uint32_t)ctx->sm_count * 8u), 256, 0, g->fwd_start,
                  (uint64_t)n + 1, dl.dptr.p);
    }
    cudaEvent_t ready = nullptr;
    cudaError_t e = cudaEventCreateWithFlags(&ready, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventRecord(ready, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->copy_stream, ready, 0);
    dl.in_flight = true;
    if (e == cudaSuccess && fwd_ptr) e = cudaMemcpyAsync(fwd_ptr, dl.dptr.p, ((size_t)n + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->copy_stream);
    if (e == cudaSuccess && u && E) e = cudaMemcpyAsync(u, dl.du.p, E * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->copy_stream);
    if (e == cudaSuccess && v && E) e = cudaMemcpyAsync(v, dl.dv.p, E * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->copy_stream);
    if (ready) cudaEventDestroy(ready);
    if (e != cudaSuccess) return ctx_fail(ctx, KOMBGPU_ECUDA, "edge list download: %s", cudaGetErrorString(e));
    return KOMBGPU_OK;
}

typedef int (*BuildFn)(kombgpu_ctx *, const uint32_t *, const uint32_t *, uint64_t, uint32_t, kombgpu_graph *);

int build_common(kombgpu_ctx *ctx, const uint32_t *a, const uint32_t *b, uint64_t count, uint32_t n, bool host_inputs,
                 BuildFn fn, kombgpu_graph **out) {
    if (!ctx) return KOMBGPU_EINVAL;
    if (!out || (count && (!a || !b))) return ctx_fail(ctx, KOMBGPU_EINVAL, "null argument");
    *out = nullptr;
    if (n >= 0xfffffffeu) return ctx_fail(ctx, KOMBGPU_EINVAL, "n_vertices too large");
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    kombgpu_graph *g = new (std::nothrow) kombgpu_graph();
    if (!g) return ctx_fail(ctx, KOMBGPU_ENOMEM, "host allocation");
    g->ctx = ctx;
    g->st.max_coreness = -1;
    const uint64_t launches0 = ctx->launches;
    int rc;
    {
        DevBuf<uint32_t> da, db;
        const uint32_t *pa = a, *pb = b;
        StageTimer timer(ctx);  // host-input copies are part of the build time when inputs are on the host
        rc = KOMBGPU_OK;
        if (host_inputs) {
            rc = upload(ctx, da, a, count);
            if (rc == KOMBGPU_OK) rc = upload(ctx, db, b, count);
            pa = da.p;
            pb = db.p;
        }
        if (rc == KOMBGPU_OK) rc = fn(ctx, pa, pb, count, n, g);
        g->st.ms_build = timer.stop();
    }
    g->st.kernel_launches = ctx->launches - launches0;
    if (rc != KOMBGPU_OK) {
        graph_release(g);
        delete g;
        return rc;
    }
    *out = g;
    return KOMBGPU_OK;
}

}  // namespace
}  // namespace kg

using namespace kg;

extern "C" {

int kombgpu_abi_version(void) { return KOMBGPU_ABI_VERSION; }

int kombgpu_ctx_create(int device, kombgpu_ctx **out) {
    if (!out) return KOMBGPU_EINVAL;
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        cudaGetLastError();
        return ctx_fail(nullptr, KOMBGPU_ENODEV, "no CUDA device available (%s); libkombgpu has no CPU fallback",
                        e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    }
    if (device < 0 || device >= count) return ctx_fail(nullptr, KOMBGPU_EINVAL, "device %d out of range [0, %d)", device, count);
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return ctx_fail(nullptr, KOMBGPU_ECUDA, "cudaGetDeviceProperties failed");
    if (prop.major != 10)
        return ctx_fail(nullptr, KOMBGPU_ENODEV, "device %d is sm_%d%d; libkombgpu is built for sm_100a (B200) only", device,
                        prop.major, prop.minor);
    if (!prop.cooperativeLaunch) return ctx_fail(nullptr, KOMBGPU_ENODEV, "device lacks cooperative launch");
    if (cudaSetDevice(device) != cudaSuccess) return ctx_fail(nullptr, KOMBGPU_ECUDA, "cudaSetDevice(%d) failed", device);
    kombgpu_ctx *ctx = new (std::nothrow) kombgpu_ctx();
    if (!ctx) return ctx_fail(nullptr, KOMBGPU_ENOMEM, "host allocation");
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    ctx->l2_bytes = (size_t)prop.l2CacheSize;
    if (cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking) != cudaSuccess) {
        delete ctx;
        return ctx_fail(nullptr, KOMBGPU_ECUDA, "cudaStreamCreate failed");
    }
    ctx->stream = ctx->own_stream;
    if (cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking) != cudaSuccess) {
        cudaStreamDestroy(ctx->own_stream);
        delete ctx;
        return ctx_fail(nullptr, KOMBGPU_ECUDA, "cudaStreamCreate failed");
    }
    if (cudaEventCreate(&ctx->ev_a) != cudaSuccess || cudaEventCreate(&ctx->ev_b) != cudaSuccess) {
        cudaStreamDestroy(ctx->copy_stream);
        cudaStreamDestroy(ctx->own_stream);
        delete ctx;
        return ctx_fail(nullptr, KOMBGPU_ECUDA, "cudaEventCreate failed");
    }
    ctx->pinned_bytes = 4096;
    if (cudaMallocHost(&ctx->pinned, ctx->pinned_bytes) != cudaSuccess) {
        ctx->pinned = nullptr;
        ctx->pinned_bytes = 0;
        cudaGetLastError();
    }
    *out = ctx;
    return KOMBGPU_OK;
}

void kombgpu_ctx_destroy(kombgpu_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    for (auto &b : ctx->arena) cudaFree(b.ptr);
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    if (ctx->ev_a) cudaEventDestroy(ctx->ev_a);
    if (ctx->ev_b) cudaEventDestroy(ctx->ev_b);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    delete ctx;
}

int kombgpu_ctx_set_stream(kombgpu_ctx *ctx, void *cuda_stream) {
    if (!ctx) return KOMBGPU_EINVAL;
    KG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->stream = static_cast<cudaStream_t>(cuda_stream);  // NULL = the legacy default stream
    return KOMBGPU_OK;
}

int kombgpu_ctx_reset_stream(kombgpu_ctx *ctx) {
    if (!ctx) return KOMBGPU_EINVAL;
    KG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->stream = ctx->own_stream;
    return KOMBGPU_OK;
}

const char *kombgpu_last_error(const kombgpu_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int kombgpu_pinned_alloc(kombgpu_ctx *ctx, uint64_t bytes, void **out) {
    if (!ctx) return KOMBGPU_EINVAL;
    if (!out) return ctx_fail(ctx, KOMBGPU_EINVAL, "null argument");
    *out = nullptr;
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    if (cudaMallocHost(out, bytes ? bytes : 1) != cudaSuccess) {
        cudaGetLastError();
        return ctx_fail(ctx, KOMBGPU_ENOMEM, "cannot page-lock %llu bytes of host memory", (unsigned long long)bytes);
    }
    return KOMBGPU_OK;
}

int kombgpu_pinned_free(kombgpu_ctx *ctx, void *ptr) {
    if (!ctx) return KOMBGPU_EINVAL;
    if (ptr) KG_CUDA(ctx, cudaFreeHost(ptr));
    return KOMBGPU_OK;
}

int kombgpu_ctx_launches(const kombgpu_ctx *ctx, uint64_t *launches) {
    if (!ctx || !launches) return KOMBGPU_EINVAL;
    *launches = ctx->launches;
    return KOMBGPU_OK;
}

int kombgpu_ctx_trim(kombgpu_ctx *ctx) {
    if (!ctx) return KOMBGPU_EINVAL;
    ws_trim(ctx);
    return KOMBGPU_OK;
}

int kombgpu_build_graph(kombgpu_ctx *ctx, const uint32_t *read_key, const uint32_t *unitig, uint64_t n_hits,
                        uint32_t n_vertices, kombgpu_graph **out) {
    return build_common(ctx, read_key, unitig, n_hits, n_vertices, true, build_from_hits, out);
}
int kombgpu_build_graph_dev(kombgpu_ctx *ctx, const uint32_t *read_key, const uint32_t *unitig, uint64_t n_hits,
                            uint32_t n_vertices, kombgpu_graph **out) {
    return build_common(ctx, read_key, unitig, n_hits, n_vertices, false, build_from_hits, out);
}
int kombgpu_graph_from_edges(kombgpu_ctx *ctx, const uint32_t *u, const uint32_t *v, uint64_t n_pairs, uint32_t n_vertices,
                             kombgpu_graph **out) {
    return build_common(ctx, u, v, n_pairs, n_vertices, true, build_from_pairs, out);
}
int kombgpu_graph_from_edges_dev(kombgpu_ctx *ctx, const uint32_t *u, const uint32_t *v, uint64_t n_pairs,
                                 uint32_t n_vertices, kombgpu_graph **out) {
    return build_common(ctx, u, v, n_pairs, n_vertices, false, build_from_pairs, out);
}

int kombgpu_graph_from_csr_dev(kombgpu_ctx *ctx, const uint64_t *row_ptr, const uint32_t *col, uint32_t n, kombgpu_graph **out) {
    if (!ctx) return KOMBGPU_EINVAL;
    if (!out || !row_ptr || n >= 0xfffffffeu) return ctx_fail(ctx, KOMBGPU_EINVAL, "bad argument");
    *out = nullptr;
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    kombgpu_graph *g = new (std::nothrow) kombgpu_graph();
    if (!g) return ctx_fail(ctx, KOMBGPU_ENOMEM, "host allocation");
    g->ctx = ctx;
    g->st.max_coreness = -1;
    const uint64_t launches0 = ctx->launches;
    int rc = adopt_csr(ctx, row_ptr, col, n, g);
    g->st.kernel_launches = ctx->launches - launches0;
    if (rc != KOMBGPU_OK) { graph_release(g); delete g; return rc; }
    *out = g;
    return KOMBGPU_OK;
}

void kombgpu_graph_destroy(kombgpu_graph *g) {
    if (!g) return;
    graph_release(g);
    delete g;
}

int kombgpu_graph_counts(const kombgpu_graph *g, uint32_t *n_vertices, uint64_t *n_edges) {
    if (!g) return KOMBGPU_EINVAL;
    if (n_vertices) *n_vertices = g->n;
    if (n_edges) *n_edges = g->n_edges;
    return KOMBGPU_OK;
}

int kombgpu_graph_edges(const kombgpu_graph *g, uint32_t *u, uint32_t *v) {
    if (!g) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = g->ctx;
    if (!u || !v) return ctx_fail(ctx, KOMBGPU_EINVAL, "null argument");
    if (g->n_edges == 0) return KOMBGPU_OK;
    if (!g->edges) return ctx_fail(ctx, KOMBGPU_ESTATE, "graph was adopted from a CSR: no canonical edge list");
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    DevBuf<uint32_t> du, dv;
    KG_ALLOC(ctx, du, g->n_edges);
    KG_ALLOC(ctx, dv, g->n_edges);
    KG_LAUNCH(ctx, unpack_edges_kernel, min(ceil_div_u64(g->n_edges, 256), (uint32_t)ctx->sm_count * 8u), 256, 0, g->edges,
              g->n_edges, du.p, dv.p);
    KG_TRY(download(ctx, du.p, u, g->n_edges));
    return download(ctx, dv.p, v, g->n_edges);
}

int kombgpu_graph_csr(const kombgpu_graph *g, uint64_t *row_ptr, uint32_t *col) {
    if (!g) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = g->ctx;
    if (!row_ptr || !col) return ctx_fail(ctx, KOMBGPU_EINVAL, "null argument");
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    KG_TRY(download(ctx, g->row_ptr, row_ptr, (size_t)g->n + 1));
    return download(ctx, g->col, col, 2 * g->n_edges);
}

int kombgpu_degree(const kombgpu_graph *g, int32_t *degree) {
    if (!g) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = g->ctx;
    if (!degree) return ctx_fail(ctx, KOMBGPU_EINVAL, "null argument");
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    return download(ctx, g->deg, degree, g->n);
}

int kombgpu_coreness(kombgpu_graph *g, int32_t *coreness) {
    if (!g) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = g->ctx;
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    if (!g->has_core) {
        const uint64_t launches0 = ctx->launches;
        StageTimer timer(ctx);
        int rc = peel_coreness(g);
        g->st.ms_peel = timer.stop();
        g->st.kernel_launches += ctx->launches - launches0;
        if (rc != KOMBGPU_OK) return rc;
    }
    if (coreness) return download(ctx, g->core, coreness, g->n);
    return KOMBGPU_OK;
}

// measurement aid (include/kombgpu_debug.h): run the peel again on a graph that already has its coreness
int kombgpu_debug_peel_again(kombgpu_graph *g) {
    if (!g) return KOMBGPU_EINVAL;
    g->has_core = false;
    return kombgpu_coreness(g, nullptr);
}

// measurement aid (include/kombgpu_debug.h): how many chunks the build reduced its pairs in
int kombgpu_debug_build_chunks(const kombgpu_graph *g, uint32_t *n_chunks) {
    if (!g || !n_chunks) return KOMBGPU_EINVAL;
    *n_chunks = g->build_chunks;
    return KOMBGPU_OK;
}

int kombgpu_corea(kombgpu_ctx *ctx, const int32_t *coreness, const int32_t *degree, uint32_t n, int key_mode, double *score) {
    if (!ctx) return KOMBGPU_EINVAL;
    if (n && (!coreness || !degree || !score)) return ctx_fail(ctx, KOMBGPU_EINVAL, "null argument");
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    DevBuf<int32_t> dc, dd;
    DevBuf<double> ds;
    KG_TRY(upload(ctx, dc, coreness, n));
    KG_TRY(upload(ctx, dd, degree, n));
    KG_ALLOC(ctx, ds, n);
    double mx = 0.0;
    KG_TRY(corea_scores(ctx, dc.p, dd.p, n, key_mode, ds.p, &mx));
    return download(ctx, ds.p, score, n);
}

int kombgpu_graph_corea(kombgpu_graph *g, int key_mode, double *score) {
    if (!g) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = g->ctx;
    if (!g->has_core) return ctx_fail(ctx, KOMBGPU_ESTATE, "kombgpu_graph_corea needs kombgpu_coreness first");
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    if (!g->score) {
        g->score = static_cast<double *>(ws_alloc(ctx, (g->n ? g->n : 1) * sizeof(double)));
        if (!g->score) return ctx_fail(ctx, KOMBGPU_ENOMEM, "score array");
    }
    {
        const uint64_t launches0 = ctx->launches;
        StageTimer timer(ctx);
        int rc = corea_scores(ctx, g->core, g->deg, g->n, key_mode, g->score, &g->max_score);
        g->st.ms_corea = timer.stop();
        g->st.kernel_launches += ctx->launches - launches0;
        if (rc != KOMBGPU_OK) return rc;
        g->has_score = true;
    }
    if (score) return download(ctx, g->score, score, g->n);
    return KOMBGPU_OK;
}

int kombgpu_graph_summary(const kombgpu_graph *g, int32_t *max_coreness, double *max_score) {
    if (!g) return KOMBGPU_EINVAL;
    if (!g->has_core) return ctx_fail(g->ctx, KOMBGPU_ESTATE, "coreness not computed yet");
    if (max_coreness) *max_coreness = g->st.max_coreness;
    if (max_score) *max_score = g->has_score ? g->max_score : 0.0;
    return KOMBGPU_OK;
}

int kombgpu_graph_analyse(kombgpu_graph *g, int key_mode) {
    KG_TRY(kombgpu_coreness(g, nullptr));
    return kombgpu_graph_corea(g, key_mode, nullptr);
}

static int graph_results_impl(kombgpu_graph *g, int key_mode, uint32_t *u, uint64_t *fwd_ptr, uint32_t *v, int32_t *degree,
                              int32_t *coreness, double *score) {
    kombgpu_ctx *ctx = g->ctx;
    const bool want_edges = v != nullptr;
    if (want_edges && g->n_edges && !g->edges) return ctx_fail(ctx, KOMBGPU_ESTATE, "graph was adopted from a CSR: no canonical edge list");
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    const uint32_t n = g->n;
    EdgeDownload dl;   // staging lives until the copy stream has drained
    // 1. edge list + degree: final after the build -> start their download on the copy stream
    int rc = KOMBGPU_OK;
    if (want_edges) rc = start_edge_download(ctx, g, g->edges, g->n_edges, n, u, fwd_ptr, v, dl);
    if (rc == KOMBGPU_OK && degree && n) {
        cudaError_t e = cudaSuccess;
        if (!dl.in_flight) {   // order the copy stream behind the build
            cudaEvent_t ready = nullptr;
            e = cudaEventCreateWithFlags(&ready, cudaEventDisableTiming);
            if (e == cudaSuccess) e = cudaEventRecord(ready, ctx->stream);
            if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->copy_stream, ready, 0);
            if (ready) cudaEventDestroy(ready);
            dl.in_flight = true;
        }
        if (e == cudaSuccess) e = cudaMemcpyAsync(degree, g->deg, n * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->copy_stream);
        if (e != cudaSuccess) rc = ctx_fail(ctx, KOMBGPU_ECUDA, "results: %s", cudaGetErrorString(e));
    }
    // 2. peel + CORE-A on the compute stream meanwhile
    if (rc == KOMBGPU_OK) rc = kombgpu_coreness(g, nullptr);
    if (rc == KOMBGPU_OK && (score || !g->has_score)) rc = kombgpu_graph_corea(g, key_mode, nullptr);
    if (rc == KOMBGPU_OK && coreness && n) rc = download(ctx, g->core, coreness, n);
    if (rc == KOMBGPU_OK && score && n) rc = download(ctx, g->score, score, n);
    cudaError_t ce = dl.in_flight ? cudaStreamSynchronize(ctx->copy_stream) : cudaSuccess;
    if (rc != KOMBGPU_OK) return rc;
    if (ce != cudaSuccess) return ctx_fail(ctx, KOMBGPU_ECUDA, "results copy stream: %s", cudaGetErrorString(ce));
    return KOMBGPU_OK;
}

int kombgpu_graph_results(kombgpu_graph *g, int key_mode, uint32_t *u, uint32_t *v, int32_t *degree, int32_t *coreness,
                          double *score) {
    if (!g) return KOMBGPU_EINVAL;
    if ((u == nullptr) != (v == nullptr)) return ctx_fail(g->ctx, KOMBGPU_EINVAL, "u and v must be given together");
    return graph_results_impl(g, key_mode, u, nullptr, v, degree, coreness, score);
}

int kombgpu_graph_results_csr(kombgpu_graph *g, int key_mode, uint64_t *fwd_ptr, uint32_t *v, int32_t *degree, int32_t *coreness,
                              double *score) {
    if (!g) return KOMBGPU_EINVAL;
    if ((fwd_ptr == nullptr) != (v == nullptr)) return ctx_fail(g->ctx, KOMBGPU_EINVAL, "fwd_ptr and v must be given together");
    return graph_results_impl(g, key_mode, nullptr, fwd_ptr, v, degree, coreness, score);
}

static int analyse_hits_impl(kombgpu_ctx *ctx, const uint32_t *read_key, const uint32_t *unitig, uint64_t n_hits, uint32_t n_vertices,
                             int key_mode, uint64_t edge_capacity, uint32_t *u, uint64_t *fwd_ptr, uint32_t *v, int32_t *degree,
                             int32_t *coreness, double *score, kombgpu_graph **out) {
    if (!out || (n_hits && (!read_key || !unitig))) return ctx_fail(ctx, KOMBGPU_EINVAL, "null argument");
    *out = nullptr;
    if (n_vertices >= 0xfffffffeu) return ctx_fail(ctx, KOMBGPU_EINVAL, "n_vertices too large");
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    kombgpu_graph *g = new (std::nothrow) kombgpu_graph();
    if (!g) return ctx_fail(ctx, KOMBGPU_ENOMEM, "host allocation");
    g->ctx = ctx;
    g->st.max_coreness = -1;
    const uint64_t launches0 = ctx->launches;
    EdgeDownload dl;   // staging of the edge list: lives until the copy stream has drained
    auto fail = [&](int rc) {
        if (dl.in_flight) cudaStreamSynchronize(ctx->copy_stream);
        graph_release(g);
        delete g;
        return rc;
    };
    int rc = KOMBGPU_OK;
    {
        StageTimer timer(ctx);
        DevBuf<uint32_t> da, db;
        rc = upload(ctx, da, read_key, n_hits);
        if (rc == KOMBGPU_OK) rc = upload(ctx, db, unitig, n_hits);
        // stage 1a: the simple edge list (final here: the CSR only adds an index over it)
        DevBuf<uint64_t> edges;
        DevBuf<uint32_t> mult;
        uint64_t E = 0;
        if (rc == KOMBGPU_OK) rc = hits_to_edges(ctx, da.p, db.p, n_hits, n_vertices, edges, &E, &g->st, &mult, &g->build_chunks);
        g->mult = mult.take();
        if (rc == KOMBGPU_OK && v && E > edge_capacity)
            rc = ctx_fail(ctx, KOMBGPU_EINVAL, "%llu edges do not fit the caller's edge buffers (%llu)", (unsigned long long)E,
                          (unsigned long long)edge_capacity);
        if (rc == KOMBGPU_OK) rc = forward_index(ctx, edges.p, E, n_vertices, &g->fwd_start);
        if (rc != KOMBGPU_OK) return fail(rc);
        // its download starts now, on the copy stream, under the rest of the build, the peel and CORE-A
        if (v) {
            rc = start_edge_download(ctx, g, edges.p, E, n_vertices, u, fwd_ptr, v, dl);
            if (rc != KOMBGPU_OK) return fail(rc);
        }
        // stage 1b: CSR
        rc = csr_from_edges(ctx, edges, E, n_vertices, g);
        g->st.ms_build = timer.stop();
        if (rc != KOMBGPU_OK) return fail(rc);
    }
    g->st.kernel_launches = ctx->launches - launches0;
    // stages 2 + 3, then the small downloads behind them on the compute stream
    rc = kombgpu_coreness(g, nullptr);
    if (rc == KOMBGPU_OK) rc = kombgpu_graph_corea(g, key_mode, nullptr);
    if (rc == KOMBGPU_OK && degree && g->n) rc = download(ctx, g->deg, degree, g->n);
    if (rc == KOMBGPU_OK && coreness && g->n) rc = download(ctx, g->core, coreness, g->n);
    if (rc == KOMBGPU_OK && score && g->n) rc = download(ctx, g->score, score, g->n);
    if (rc != KOMBGPU_OK) return fail(rc);
    if (dl.in_flight) {
        cudaError_t ce = cudaStreamSynchronize(ctx->copy_stream);
        dl.in_flight = false;
        if (ce != cudaSuccess) return fail(ctx_fail(ctx, KOMBGPU_ECUDA, "analyse_hits copy stream: %s", cudaGetErrorString(ce)));
    }
    *out = g;
    return KOMBGPU_OK;
}

int kombgpu_analyse_hits(kombgpu_ctx *ctx, const uint32_t *read_key, const uint32_t *unitig, uint64_t n_hits, uint32_t n_vertices,
                         int key_mode, uint64_t edge_capacity, uint32_t *u, uint32_t *v, int32_t *degree, int32_t *coreness,
                         double *score, kombgpu_graph **out) {
    if (!ctx) return KOMBGPU_EINVAL;
    if ((u == nullptr) != (v == nullptr)) return ctx_fail(ctx, KOMBGPU_EINVAL, "u and v must be given together");
    return analyse_hits_impl(ctx, read_key, unitig, n_hits, n_vertices, key_mode, edge_capacity, u, nullptr, v, degree, coreness, score, out);
}

int kombgpu_analyse_hits_csr(kombgpu_ctx *ctx, const uint32_t *read_key, const uint32_t *unitig, uint64_t n_hits, uint32_t n_vertices,
                             int key_mode, uint64_t edge_capacity, uint64_t *fwd_ptr, uint32_t *v, int32_t *degree, int32_t *coreness,
                             double *score, kombgpu_graph **out) {
    if (!ctx) return KOMBGPU_EINVAL;
    if ((fwd_ptr == nullptr) != (v == nullptr)) return ctx_fail(ctx, KOMBGPU_EINVAL, "fwd_ptr and v must be given together");
    return analyse_hits_impl(ctx, read_key, unitig, n_hits, n_vertices, key_mode, edge_capacity, nullptr, fwd_ptr, v, degree, coreness, score, out);
}

int kombgpu_graph_edges_csr(const kombgpu_graph *g, uint64_t *fwd_ptr, uint32_t *v) {
    if (!g) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = g->ctx;
    if (!fwd_ptr || (g->n_edges && !v)) return ctx_fail(ctx, KOMBGPU_EINVAL, "null argument");
    if (!g->fwd_start) return ctx_fail(ctx, KOMBGPU_ESTATE, "graph was adopted from a CSR: no canonical edge list");
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    EdgeDownload dl;
    int rc = start_edge_download(ctx, g, g->edges, g->n_edges, g->n, nullptr, fwd_ptr, v, dl);
    cudaError_t ce = dl.in_flight ? cudaStreamSynchronize(ctx->copy_stream) : cudaSuccess;
    if (rc != KOMBGPU_OK) return rc;
    if (ce != cudaSuccess) return ctx_fail(ctx, KOMBGPU_ECUDA, "edge list download: %s", cudaGetErrorString(ce));
    return KOMBGPU_OK;
}

int kombgpu_graph_edge_multiplicity(const kombgpu_graph *g, uint32_t *mult) {
    if (!g) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = g->ctx;
    if (g->n_edges && !mult) return ctx_fail(ctx, KOMBGPU_EINVAL, "null argument");
    if (g->n_edges == 0) return KOMBGPU_OK;
    if (!g->mult) return ctx_fail(ctx, KOMBGPU_ESTATE, "graph was adopted from a CSR: no edge multiplicities");
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    return download(ctx, g->mult, mult, g->n_edges);
}

int kombgpu_graph_stats(const kombgpu_graph *g, kombgpu_stats *out) {
    if (!g || !out) return KOMBGPU_EINVAL;
    *out = g->st;
    return KOMBGPU_OK;
}

int kombgpu_graph_device_arrays(const kombgpu_graph *g, const uint64_t **row_ptr, const uint32_t **col,
                                const uint64_t **edges_packed, const int32_t **degree, const int32_t **coreness,
                                const double **score) {
    if (!g) return KOMBGPU_EINVAL;
    if (row_ptr) *row_ptr = g->row_ptr;
    if (col) *col = g->col;
    if (edges_packed) *edges_packed = g->edges;
    if (degree) *degree = g->deg;
    if (coreness) *coreness = g->has_core ? g->core : nullptr;
    if (score) *score = g->has_score ? g->score : nullptr;
    return KOMBGPU_OK;
}

}  // extern "C"
