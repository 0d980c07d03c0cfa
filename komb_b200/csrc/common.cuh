// common.cuh — context, workspace arena, error plumbing and small device helpers
// shared by every translation unit of libkombgpu.so (sm_100a only).
#pragma once

#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>
#include <string>
#include <vector>

#include "kombgpu.h"

namespace kg {

constexpr int kWarp = 32;
constexpr uint32_t kFullMask = 0xffffffffu;

// ---------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------
struct ArenaBlock {
    void *ptr;
    size_t bytes;
    bool in_use;
};

}  // namespace kg

struct kombgpu_ctx {
    int device = -1;
    int sm_count = 0;
    size_t l2_bytes = 0;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;  // downloads that overlap compute (kombgpu_graph_results)
    std::string err;
    std::vector<kg::ArenaBlock> arena;  // cached device workspace, reused across calls
    uint64_t launches = 0;              // kernels launched through this context
    void *pinned = nullptr;             // small pinned staging area for scalar read-backs
    size_t pinned_bytes = 0;
    bool sort_attr_set = false;         // function attributes are per device: set once per context (sort.cu)
    bool corea_attr_set = false;        // same for the CORE-A pair histogram (corea.cu)
    bool peer_attr_set = false;         // same for the partitioned peel kernel (ppeel.cu)
    cudaEvent_t ev_a = nullptr, ev_b = nullptr;   // stage timers (capi.cu StageTimer): created once
};

namespace kg {

int ctx_fail(kombgpu_ctx *ctx, int code, const char *fmt, ...);

// Stream-ordered workspace: every kernel of a context runs on ctx->stream, so a
// block handed back with ws_free may be reused by the next launch immediately.
void *ws_alloc(kombgpu_ctx *ctx, size_t bytes);
void ws_free(kombgpu_ctx *ctx, void *p);
// hand a block back to the device at once (a buffer that keeps growing, so the cache could never reuse it)
void ws_release(kombgpu_ctx *ctx, void *p);
void ws_trim(kombgpu_ctx *ctx);

// RAII holder for workspace blocks.
template <typename T>
struct DevBuf {
    kombgpu_ctx *ctx = nullptr;
    T *p = nullptr;
    size_t count = 0;
    DevBuf() = default;
    DevBuf(kombgpu_ctx *c, size_t n) { alloc(c, n); }
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    DevBuf(DevBuf &&o) noexcept : ctx(o.ctx), p(o.p), count(o.count) { o.p = nullptr; o.count = 0; }
    DevBuf &operator=(DevBuf &&o) noexcept {
        if (this != &o) { release(); ctx = o.ctx; p = o.p; count = o.count; o.p = nullptr; o.count = 0; }
        return *this;
    }
    ~DevBuf() { release(); }
    bool alloc(kombgpu_ctx *c, size_t n) {
        release();
        ctx = c;
        count = n;
        p = static_cast<T *>(ws_alloc(c, (n ? n : 1) * sizeof(T)));
        return p != nullptr;
    }
    void release() {
        if (p) ws_free(ctx, p);
        p = nullptr;
        count = 0;
    }
    T *take() { T *q = p; p = nullptr; count = 0; return q; }
    explicit operator bool() const { return p != nullptr; }
};

#define KG_CUDA(ctx, call)                                                                   \
    do {                                                                                     \
        cudaError_t kg_e_ = (call);                                                          \
        if (kg_e_ != cudaSuccess)                                                            \
            return kg::ctx_fail((ctx), KOMBGPU_ECUDA, "%s:%d %s: %s", __FILE__, __LINE__, #call, \
                                cudaGetErrorString(kg_e_));                                  \
    } while (0)

#define KG_TRY(expr)                  \
    do {                              \
        int kg_rc_ = (expr);          \
        if (kg_rc_ != KOMBGPU_OK) return kg_rc_; \
    } while (0)

#define KG_ALLOC(ctx, buf, n)                                                               \
    do {                                                                                    \
        if (!(buf).alloc((ctx), (n)))                                                       \
            return kg::ctx_fail((ctx), KOMBGPU_ENOMEM, "%s:%d device workspace of %zu bytes", \
                                __FILE__, __LINE__, (size_t)(n) * sizeof(*(buf).p));        \
    } while (0)

// Launch bookkeeping: every kernel launch goes through KG_LAUNCH so that
// kombgpu_stats.kernel_launches is a real count.
#define KG_LAUNCH(ctx, kernel, grid, block, smem, ...)                                      \
    do {                                                                                    \
        kernel<<<(grid), (block), (smem), (ctx)->stream>>>(__VA_ARGS__);                    \
        (ctx)->launches++;                                                                  \
        cudaError_t kg_e_ = cudaPeekAtLastError();                                          \
        if (kg_e_ != cudaSuccess)                                                           \
            return kg::ctx_fail((ctx), KOMBGPU_ECUDA, "%s:%d launch %s: %s", __FILE__, __LINE__, \
                                #kernel, cudaGetErrorString(kg_e_));                        \
    } while (0)

inline uint32_t ceil_div_u64(uint64_t a, uint64_t b) { return (uint32_t)((a + b - 1) / b); }

inline int bits_for(uint64_t max_value) {  // number of bits needed to represent max_value
    int b = 0;
    while (max_value) { ++b; max_value >>= 1; }
    return b;
}

// Small read-backs (counters, totals, the peel's state) go through a copy KERNEL that stores into the context's
// page-locked staging area (device-accessible under UVA), not through cudaMemcpy: a DMA copy would queue on the
// device-to-host copy engine behind a bulk download that is in flight on the copy stream (the edge list, 5 ms for
// cfg2) and stall the compute stream's host for that long.
int small_read_back(kombgpu_ctx *ctx, const void *dev, void *host, size_t bytes);   // capi.cu; bytes <= ctx->pinned_bytes

// read back `count` elements of T from the device
template <typename T>
int read_back(kombgpu_ctx *ctx, const T *dev, T *host, size_t count) {
    size_t bytes = count * sizeof(T);
    if (bytes == 0) return KOMBGPU_OK;
    if (bytes <= ctx->pinned_bytes) return small_read_back(ctx, dev, host, bytes);
    KG_CUDA(ctx, cudaMemcpyAsync(host, dev, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    KG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return KOMBGPU_OK;
}

// ---------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------
#ifdef __CUDACC__

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31; }
__device__ __forceinline__ uint32_t lanemask_lt() {
    uint32_t m;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}

// L2-coherent loads (skip the non-coherent L1): for data other CTAs update
// with atomics inside the same launch.
__device__ __forceinline__ int32_t ld_cg_s32(const int32_t *p) { return __ldcg(p); }
__device__ __forceinline__ uint32_t ld_cg_u32(const uint32_t *p) { return __ldcg(p); }
__device__ __forceinline__ uint32_t ld_volatile_u32(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
// streaming 16-byte load / store: touched once, keep it out of L1
__device__ __forceinline__ uint4 ld_stream_u4(const uint4 *p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}

template <typename T>
__device__ __forceinline__ T warp_incl_scan_add(T v) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        T t = __shfl_up_sync(kFullMask, v, o);
        if (lane_id() >= (uint32_t)o) v += t;
    }
    return v;
}

template <typename T>
__device__ __forceinline__ T warp_reduce_add(T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFullMask, v, o);
    return v;
}

template <typename T>
__device__ __forceinline__ T warp_reduce_max(T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { T t = __shfl_xor_sync(kFullMask, v, o); v = t > v ? t : v; }
    return v;
}

template <typename T>
__device__ __forceinline__ T warp_reduce_min(T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { T t = __shfl_xor_sync(kFullMask, v, o); v = t < v ? t : v; }
    return v;
}

// Block-wide exclusive prefix sum of one value per thread.  `smem` holds
// THREADS/32 + 1 elements.  Returns the exclusive prefix; *total = block sum.
template <typename T, int THREADS>
__device__ __forceinline__ T block_excl_scan_add(T v, T *smem, T *total) {
    constexpr int W = THREADS / 32;
    const uint32_t lane = lane_id(), warp = threadIdx.x >> 5;
    T incl = warp_incl_scan_add(v);
    if (lane == 31) smem[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        T w = lane < W ? smem[lane] : T(0);
        T wi = warp_incl_scan_add(w);
        if (lane < W) smem[lane] = wi - w;
        if (lane == W - 1) smem[W] = wi;
    }
    __syncthreads();
    T res = smem[warp] + incl - v;
    *total = smem[W];
    __syncthreads();
    return res;
}

#endif  // __CUDACC__

}  // namespace kg
