// prank.cuh — the rank-level device primitives of the peels that exchange logs over peer memory (ppeel.cu, ponion.cu):
// scoped loads and stores, the global timer, the barrier of one rank's CTAs, the read of a peer's log entry and the
// publish of the own log, each with the watchdog that turns a wait that never ends into an error.
//
// The state types they take (S) have the fields these functions name: bar_count, bar_gen, error (and for the publish
// published, log_cnt); the rank descriptors (R) have world, rank, log_local[], log_peer[].
#pragma once

#include "dgraph.cuh"

namespace kg {
namespace {

constexpr unsigned long long kPeelWatchdogNs = 20ull * 1000000000ull;
constexpr unsigned long long kTagShift = 40, kValMask = (1ull << 40) - 1;

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
            atomicCAS(&st->error, 0u, 2u);
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
                    atomicCAS(&st->error, 0u, 1u);
                    break;
                }
            }
        }
        __threadfence();
    }
    __syncthreads();
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

}  // namespace
}  // namespace kg
