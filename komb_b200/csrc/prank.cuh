// prank.cuh — what the persistent rank kernels of the partitioned path (ppeel.cu, apeel.cu, ponion.cu) share.
//   device   scoped loads and stores, the global timer, the barrier of one rank's CTAs, the wait for CTA 0's plan, the
//            read of a peer's log entry and the publish of the own log, each with the watchdog that turns a wait that
//            never ends into an error code
//   host     the CTAs per rank and the launch: one grid per GPU, or one grid for every rank when they share a device
//
// The state types the device functions take (S) have the fields they name: bar_count, bar_gen, error (and for the
// publish published, log_cnt); the rank descriptors (R) have world, rank, log_local[], log_peer[].
#pragma once

#include <vector>

#include "dgraph.cuh"

namespace kg {
namespace {

constexpr unsigned long long kPeelWatchdogNs = 20ull * 1000000000ull;
constexpr unsigned long long kTagShift = 40, kValMask = (1ull << 40) - 1;

// the error word of a rank kernel's state: the first failure stands
enum : uint32_t { kErrBarrier = 1, kErrPeers = 2, kErrBadEntry = 4, kErrFull = 5 };
inline const char *rank_error_text(unsigned long long e) {
    switch (e) {
        case kErrBarrier: return "watchdog inside a rank";
        case kErrPeers: return "watchdog between the ranks";
        case kErrBadEntry: return "bad log or pool entry";
        case kErrFull: return "list or pool full";
        default: return "unknown error";
    }
}

__device__ __forceinline__ unsigned long long ld_relaxed_sys(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long ld_acq_gpu(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_rel_gpu(unsigned long long *p, unsigned long long v) {
    asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void st_relaxed_sys(unsigned long long *p, unsigned long long v) {
    asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long pglobal_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// A log entry of a peer is valid as soon as it differs from kLogEmpty (the logs are cleared before the peel and every slot
// is written once): the length a peer publishes may overtake the entries themselves on the wire, so no fence or
// acknowledgement round trip stands between copying ids and announcing them.
constexpr uint32_t kLogEmpty = 0xffffffffu;
template <class S>
__device__ __forceinline__ uint32_t log_read(const uint32_t *slot, S *st) {
    uint32_t x = *reinterpret_cast<const volatile uint32_t *>(slot);
    if (x != kLogEmpty) return x;
    const unsigned long long t0 = pglobal_ns();
    uint32_t spins = 0;
    while ((x = *reinterpret_cast<const volatile uint32_t *>(slot)) == kLogEmpty) {
        if ((++spins & 1023u) == 0 && (*(volatile uint32_t *)&st->error || pglobal_ns() - t0 > kPeelWatchdogNs)) {
            atomicCAS(&st->error, 0u, (uint32_t)kErrPeers);
            break;
        }
    }
    return x;
}

// barrier of one rank's CTAs.  sys_fence: the CTAs stored into peer memory before it, and those stores must be
// visible at the peer before the leader publishes this rank's counts after it.
template <class S>
__device__ __forceinline__ void rank_barrier(S *st, uint32_t ctas, unsigned long long &gen, bool sys_fence) {
    __syncthreads();
    if (threadIdx.x == 0) {
        if (sys_fence) __threadfence_system(); else __threadfence();
        ++gen;
        const unsigned long long arrived = atomicAdd(&st->bar_count, 1ull) + 1ull;
        if (arrived == gen * ctas) {
            st_rel_gpu(&st->bar_gen, gen);
        } else {
            const unsigned long long t0 = pglobal_ns();
            uint32_t spins = 0;
            while (ld_acq_gpu(&st->bar_gen) < gen) {
                if ((++spins & 4095u) == 0 && (*(volatile uint32_t *)&st->error || pglobal_ns() - t0 > kPeelWatchdogNs)) {
                    atomicCAS(&st->error, 0u, (uint32_t)kErrBarrier);
                    break;
                }
            }
        }
        __threadfence();
    }
    __syncthreads();
}

// every CTA learns what CTA 0 released for step t: the flags of (t << 8) | flags in *word, or kDone after a watchdog
template <uint32_t kDone, class S>
__device__ __forceinline__ uint32_t wait_plan(unsigned long long *word, uint32_t t, S *st, uint32_t *s_bcast) {
    if (threadIdx.x == 0) {
        const unsigned long long t0 = pglobal_ns();
        uint32_t spins = 0, res = 0;
        while (true) {
            const unsigned long long w = ld_acq_gpu(word);
            if ((uint32_t)(w >> 8) == t) { res = (uint32_t)(w & 0xffu); break; }
            if ((++spins & 4095u) == 0 && (*(volatile uint32_t *)&st->error || pglobal_ns() - t0 > kPeelWatchdogNs)) {
                atomicCAS(&st->error, 0u, (uint32_t)kErrBarrier);
                res = kDone;
                break;
            }
        }
        *s_bcast = res;
    }
    __syncthreads();
    const uint32_t r = *s_bcast;
    __syncthreads();
    return r;
}

// PUBLISH: copy the new part of the own log into every peer's copy (thread gthread of nthreads)
template <class R_t, class S>
__device__ __forceinline__ void publish_stage(const R_t &R, S *st, uint32_t gthread, uint32_t nthreads) {
    const uint32_t lo = __ldcg(&st->published), hi = __ldcg(&st->log_cnt);
    const uint32_t *src = R.log_local[R.rank];
    for (int p = 0; p < R.world; ++p) {
        if (p == R.rank) continue;
        uint32_t *dst = R.log_peer[p];
        for (uint32_t i = lo + gthread; i < hi; i += nthreads) dst[i] = __ldcg(&src[i]);
    }
}

// ---- host

// CTAs per rank of a persistent rank kernel: as many as are resident at once, shared by the ranks of one device
template <class K>
int rank_ctas(kombgpu_ctx *ctx, const kombgpu_comm *c, K kernel, int threads, uint32_t min_ctas, uint32_t *ctas_per_rank) {
    int per_sm = 0;
    KG_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, 0));
    if (per_sm < 1) return ctx_fail(ctx, KOMBGPU_ECUDA, "a persistent rank kernel does not fit on an SM");
    const int resident = per_sm * ctx->sm_count;
    *ctas_per_rank = c->same_device ? (uint32_t)(resident / c->world) : (uint32_t)resident;
    if (*ctas_per_rank < min_ctas) return ctx_fail(ctx, KOMBGPU_EINVAL, "too many ranks on one device");
    return KOMBGPU_OK;
}

// Runs kernel(descriptors, ctas_per_rank) to its end, a cooperative grid of ctas_per_rank CTAs per rank, and returns
// the CUDA status.  With a GPU per rank every rank launches its own grid.  Ranks that share one device (emulation)
// run inside ONE grid, since kernels of different ranks must never wait for one another on the same GPU: every rank
// hands its descriptor to rank 0's thread (LocalGroup::slot), which launches for all of them.  Every rank passes the
// three group barriers, whatever failed.  ms_kernel (optional): the kernel's time, set on the rank that launched.
template <class D, class K>
cudaError_t launch_ranks(kombgpu_comm *c, K kernel, int threads, uint32_t ctas_per_rank, const D &mine, D *desc_dev, float *ms_kernel) {
    kombgpu_ctx *ctx = c->ctx;
    auto launch = [&](const D *desc, int n_ranks) -> cudaError_t {
        cudaError_t e = cudaMemcpyAsync(desc_dev, desc, sizeof(D) * n_ranks, cudaMemcpyHostToDevice, ctx->stream);
        const D *dp = desc_dev;
        uint32_t cpr = ctas_per_rank;
        void *args[] = {(void *)&dp, (void *)&cpr};
        if (e != cudaSuccess) return e;
        if (ms_kernel) {
            EvTimer timer(ctx);
            e = cudaLaunchCooperativeKernel((void *)kernel, dim3(ctas_per_rank * n_ranks), dim3(threads), args, 0, ctx->stream);
            if (e == cudaSuccess) *ms_kernel = timer.lap();
        } else {
            e = cudaLaunchCooperativeKernel((void *)kernel, dim3(ctas_per_rank * n_ranks), dim3(threads), args, 0, ctx->stream);
        }
        ctx->launches++;
        return e == cudaSuccess ? cudaStreamSynchronize(ctx->stream) : e;
    };
    if (!c->same_device) return launch(&mine, 1);
    LocalGroup *grp = c->group;
    grp->slot[c->rank] = &mine;
    bool met = comm_group_barrier(c) == KOMBGPU_OK;
    cudaError_t le = cudaSuccess;
    if (c->rank == 0) {
        std::vector<D> all(c->world);
        for (int q = 0; met && q < c->world; ++q) all[q] = *static_cast<const D *>(grp->slot[q]);
        le = met ? launch(all.data(), c->world) : cudaErrorLaunchFailure;
        grp->slot_rc = le == cudaSuccess ? 0 : 1;
    }
    met = comm_group_barrier(c) == KOMBGPU_OK && met;
    if (!met || grp->slot_rc) le = cudaErrorLaunchFailure;
    met = comm_group_barrier(c) == KOMBGPU_OK && met;   // slot_rc was read by everyone before the next use
    return met ? le : cudaErrorLaunchFailure;
}

}  // namespace
}  // namespace kg
