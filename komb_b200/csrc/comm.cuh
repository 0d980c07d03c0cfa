// comm.cuh — the communicator of the multi-GPU path: one rank per GPU, ranks talk through PEER MEMORY (NVLink /
// NVSwitch), not through a collective library.
//
//   symmetric heap   every rank allocates the same sequence of buffers; a rank holds, for each buffer, the pointer
//                    of every peer's copy mapped into its own address space (cudaIpc between processes, plain
//                    peer access between the devices of one process).  Kernels store to / load from those pointers.
//   exchange         an all-gather of a few 64-bit words per rank that doubles as the barrier between phases: one
//                    tiny kernel stores the words and an epoch flag into every peer's control block, then waits
//                    for every peer's flag (stream-ordered: no host round trip except to read the result).
//   bootstrap        the only thing a host has to provide is an all-gather of small byte blobs between the ranks
//                    (kombgpu_allgather_fn: torch.distributed / MPI between processes; built in for the ranks of
//                    one process).
// Ranks that share ONE device (tests on a one-GPU box) never wait for one another on the device: kernels that
// spin on a peer's flag are only safe when every rank has its own GPU, so in that case the exchange is done by the
// host threads (stream sync + host barrier) and the peel runs all ranks inside one cooperative grid.
#pragma once

#include <condition_variable>
#include <mutex>
#include <vector>

#include "common.cuh"

namespace kg {

constexpr int kMaxRanks = 16;
constexpr int kCtlWords = 24;   // 64-bit words one rank can publish per exchange

template <typename T>
struct PeerPtrs {
    T *p[kMaxRanks];
};

// control block, one per rank, in symmetric memory (zero-initialised)
struct CtlBlock {
    unsigned long long flag[2][kMaxRanks];                // flag[parity][src] = epoch of src's last exchange of that parity
    unsigned long long data[2][kMaxRanks][kCtlWords];     // words published by src
};

// the ranks of one process (one host thread per rank): bootstrap all-gather and host barrier
struct LocalGroup {
    int world = 0;
    std::mutex mu;
    std::condition_variable cv;
    int arrived = 0;
    uint64_t generation = 0;
    std::vector<unsigned char> blob;   // world x bytes_per_rank of the all-gather in flight
    bool broken = false;               // a rank failed: every waiter gives up
    int refs = 0;
    // same-device emulation: the descriptors the ranks hand to the one thread that launches a persistent rank kernel
    // for all of them (launch_ranks in prank.cuh, for ppeel.cu, apeel.cu and ponion.cu)
    const void *slot[kMaxRanks] = {};
    int slot_rc = 0;
};

struct SymSegment {
    void *local = nullptr;
    void *peer[kMaxRanks] = {};
    bool ipc_opened[kMaxRanks] = {};
    size_t bytes = 0, used = 0;
};

}  // namespace kg

struct kombgpu_comm {
    kombgpu_ctx *ctx = nullptr;
    int rank = 0, world = 1;
    kombgpu_allgather_fn allgather = nullptr;
    void *user = nullptr;
    kg::LocalGroup *group = nullptr;      // set for the ranks of one process
    bool same_device = false;             // every rank on one device: host-side exchange, one-grid peel
    bool device_wait_ok = true;           // kernels may spin on peers' flags (false under same_device)
    size_t seg_bytes = 0;                 // default size of a new heap segment
    std::vector<kg::SymSegment> segs;
    kg::CtlBlock *ctl = nullptr;          // this rank's control block (in segment 0)
    kg::PeerPtrs<kg::CtlBlock> ctl_peers{};
    uint64_t epoch = 0;
    unsigned long long *xchg_out = nullptr;   // pinned host: result of the last exchange [world][kCtlWords]
    uint64_t sym_high_water = 0;
};

namespace kg {

// collective: every rank calls it with the same `bytes`; returns the local buffer, peers->p[q] = rank q's copy
// (peers->p[rank] = local).  Stack discipline: sym_mark() / sym_release(mark).
template <typename T>
int sym_alloc(kombgpu_comm *c, size_t count, T **local, PeerPtrs<T> *peers);
int sym_alloc_bytes(kombgpu_comm *c, size_t bytes, void **local, void **peers /* [kMaxRanks] */);
struct SymMark { size_t seg; size_t used; };
SymMark sym_mark(const kombgpu_comm *c);
void sym_release(kombgpu_comm *c, SymMark m);

// all-gather of k <= kCtlWords words per rank + barrier, ordered on the context's stream; out[q * k + j] on the host
int comm_exchange(kombgpu_comm *c, const unsigned long long *vals, int k, unsigned long long *out);
// comm_exchange of k < kCtlWords words per rank that also carries every rank's status rc: a rank that failed returns
// its own code, the others fail with the code of the first failing rank.  The collectives of the partitioned path meet
// through these two, and a rank that failed locally keeps making the same calls as its peers up to the next one.
int exchange_rc(kombgpu_comm *c, int rc, const unsigned long long *vals, int k, unsigned long long *out);
inline int barrier_rc(kombgpu_comm *c, int rc) { return exchange_rc(c, rc, nullptr, 0, nullptr); }
// a status that collects the steps every rank makes whatever failed before (sym_alloc): the first failure stands
inline int first_rc(int rc, int next) { return rc != KOMBGPU_OK ? rc : next; }
// host-side bootstrap all-gather (slow path: setup only)
int comm_bootstrap_allgather(kombgpu_comm *c, const void *send, void *recv, size_t bytes_per_rank);
// host barrier of the ranks of one process (same-device emulation only)
int comm_group_barrier(kombgpu_comm *c);
// sum / max of one value over the ranks, via comm_exchange
int comm_allreduce_sum(kombgpu_comm *c, unsigned long long v, unsigned long long *out);

struct SymRewind {   // gives the symmetric heap back to a mark when the scope ends, on every return path
    kombgpu_comm *c;
    SymMark mark;
    ~SymRewind() { sym_release(c, mark); }
};

struct EvTimer {   // CUDA-event split timer on the context's stream
    kombgpu_ctx *ctx;
    cudaEvent_t a = nullptr, b = nullptr;
    explicit EvTimer(kombgpu_ctx *c) : ctx(c) { cudaEventCreate(&a); cudaEventCreate(&b); cudaEventRecord(a, ctx->stream); }
    float lap() {
        float ms = 0.f;
        cudaEventRecord(b, ctx->stream);
        cudaEventSynchronize(b);
        cudaEventElapsedTime(&ms, a, b);
        cudaEventRecord(a, ctx->stream);
        return ms;
    }
    ~EvTimer() { cudaEventDestroy(a); cudaEventDestroy(b); }
};

template <typename T>
int sym_alloc(kombgpu_comm *c, size_t count, T **local, PeerPtrs<T> *peers) {
    void *l = nullptr;
    void *pp[kMaxRanks] = {};
    int rc = sym_alloc_bytes(c, (count ? count : 1) * sizeof(T), &l, pp);
    if (rc != KOMBGPU_OK) return rc;
    *local = static_cast<T *>(l);
    if (peers)
        for (int q = 0; q < kMaxRanks; ++q) peers->p[q] = static_cast<T *>(pp[q]);
    return KOMBGPU_OK;
}

}  // namespace kg
