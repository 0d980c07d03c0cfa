// comm.cu — communicator of the multi-GPU path (see comm.cuh): bootstrap, symmetric heap over peer memory,
// stream-ordered exchange (all-gather of a few words + barrier).
//
// Replaces nothing in the reference (komb2 is a single process on one host, src/komb2.cpp); it is the plumbing under
// the partitioned build / peel / CORE-A of SURVEY.md section 8(e).
#include <unistd.h>

#include <cstring>
#include <new>

#include "comm.cuh"

namespace kg {
namespace {

constexpr unsigned long long kExchangeWatchdogNs = 30ull * 1000000000ull;

struct ExchangeWords {
    unsigned long long w[kCtlWords];
};

__device__ __forceinline__ unsigned long long ld_acquire_sys_u64(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys_u64(unsigned long long *p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long comm_global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// thread q: publish my words in rank q's control block, then wait for rank q's words in mine.
// out[q * k + j]; out[world * k] = 0 on success, 1 when a peer never showed up (watchdog).
__global__ void exchange_kernel(PeerPtrs<CtlBlock> peers, int rank, int world, unsigned long long epoch, ExchangeWords vals, int k,
                                unsigned long long *out) {
    const int q = threadIdx.x;
    const int par = (int)(epoch & 1ull);
    bool failed = false;
    if (q < world) {
        CtlBlock *dst = peers.p[q];
        for (int j = 0; j < k; ++j) dst->data[par][rank][j] = vals.w[j];
        __threadfence_system();   // the words (and everything this stream wrote to rank q before) are visible before the flag
        st_release_sys_u64(&dst->flag[par][rank], epoch);
        const CtlBlock *mine = peers.p[rank];
        const unsigned long long t0 = comm_global_ns();
        unsigned int spins = 0;
        while (ld_acquire_sys_u64(&mine->flag[par][q]) != epoch) {
            if ((++spins & 1023u) == 0 && comm_global_ns() - t0 > kExchangeWatchdogNs) { failed = true; break; }
        }
        if (!failed)
            for (int j = 0; j < k; ++j) out[q * k + j] = *(const volatile unsigned long long *)&mine->data[par][q][j];
    }
    const unsigned int any_failed = __ballot_sync(0xffffffffu, failed);
    if (threadIdx.x == 0) out[world * k] = any_failed ? 1ull : 0ull;
}

struct BootInfo {
    int pid;
    int device;
    int can_ipc;
    int in_group;
    unsigned long long host_hash;
    char bus_id[32];
};

unsigned long long hostname_hash() {
    char name[256] = {0};
    gethostname(name, sizeof(name) - 1);
    unsigned long long h = 1469598103934665603ull;
    for (const char *p = name; *p; ++p) { h ^= (unsigned char)*p; h *= 1099511628211ull; }
    return h;
}

int group_barrier(LocalGroup *g) {
    std::unique_lock<std::mutex> lk(g->mu);
    if (g->broken) return KOMBGPU_ESTATE;
    const uint64_t gen = g->generation;
    if (++g->arrived == g->world) {
        g->arrived = 0;
        ++g->generation;
        g->cv.notify_all();
    } else {
        g->cv.wait(lk, [&] { return g->generation != gen || g->broken; });
    }
    return g->broken ? KOMBGPU_ESTATE : KOMBGPU_OK;
}

// the bootstrap all-gather of the ranks of one process
int group_allgather(void *user, const void *send, void *recv, uint64_t bytes) {
    kombgpu_comm *c = static_cast<kombgpu_comm *>(user);
    LocalGroup *g = c->group;
    {
        std::lock_guard<std::mutex> lk(g->mu);
        if (g->blob.size() < (size_t)g->world * bytes) g->blob.resize((size_t)g->world * bytes);
        memcpy(g->blob.data() + (size_t)c->rank * bytes, send, bytes);
    }
    if (group_barrier(g) != KOMBGPU_OK) return -1;
    memcpy(recv, g->blob.data(), (size_t)g->world * bytes);   // nobody writes between the two barriers
    if (group_barrier(g) != KOMBGPU_OK) return -1;
    return 0;
}

int new_segment(kombgpu_comm *c, size_t bytes) {
    kombgpu_ctx *ctx = c->ctx;
    SymSegment seg;
    seg.bytes = bytes;
    cudaError_t e = cudaMalloc(&seg.local, bytes);
    if (e != cudaSuccess) {
        cudaGetLastError();
        ws_trim(ctx);   // give cached workspace back and retry once
        e = cudaMalloc(&seg.local, bytes);
    }
    // every rank reports success or failure before anyone opens a handle, so a failed rank cannot strand its peers
    struct SegMsg {
        int ok;
        int pad;
        void *ptr;
        cudaIpcMemHandle_t handle;
    } mine{}, all[kMaxRanks];
    mine.ok = e == cudaSuccess ? 1 : 0;
    mine.ptr = seg.local;
    if (e != cudaSuccess) cudaGetLastError();
    if (mine.ok && !c->group && c->world > 1) {
        cudaError_t he = cudaIpcGetMemHandle(&mine.handle, seg.local);
        if (he != cudaSuccess) { cudaGetLastError(); mine.ok = 0; }
    }
    if (comm_bootstrap_allgather(c, &mine, all, sizeof(SegMsg)) != KOMBGPU_OK) {
        if (seg.local) cudaFree(seg.local);
        return ctx_fail(ctx, KOMBGPU_ESTATE, "communicator bootstrap failed while growing the symmetric heap");
    }
    bool ok = true;
    for (int q = 0; q < c->world; ++q) ok = ok && all[q].ok;
    if (!ok) {
        if (seg.local) cudaFree(seg.local);
        return ctx_fail(ctx, KOMBGPU_ENOMEM, "symmetric heap: a rank could not allocate or export %zu bytes", bytes);
    }
    for (int q = 0; q < c->world; ++q) {
        if (q == c->rank) { seg.peer[q] = seg.local; continue; }
        if (c->group) {
            seg.peer[q] = all[q].ptr;   // same process: the peer's pointer is valid here (peer access enabled at creation)
        } else {
            cudaError_t oe = cudaIpcOpenMemHandle(&seg.peer[q], all[q].handle, cudaIpcMemLazyEnablePeerAccess);
            if (oe != cudaSuccess) {
                cudaGetLastError();
                for (int r = 0; r < q; ++r)
                    if (seg.ipc_opened[r]) cudaIpcCloseMemHandle(seg.peer[r]);
                cudaFree(seg.local);
                return ctx_fail(ctx, KOMBGPU_ECUDA, "cudaIpcOpenMemHandle (rank %d -> rank %d): %s", c->rank, q, cudaGetErrorString(oe));
            }
            seg.ipc_opened[q] = true;
        }
    }
    KG_CUDA(ctx, cudaMemsetAsync(seg.local, 0, bytes, ctx->stream));
    KG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    c->segs.push_back(seg);
    // nobody may store into a peer's new segment before that peer has cleared it
    int token = 1, tokens[kMaxRanks];
    if (comm_bootstrap_allgather(c, &token, tokens, sizeof(int)) != KOMBGPU_OK)
        return ctx_fail(ctx, KOMBGPU_ESTATE, "communicator bootstrap barrier failed");
    return KOMBGPU_OK;
}

}  // namespace

int comm_bootstrap_allgather(kombgpu_comm *c, const void *send, void *recv, size_t bytes_per_rank) {
    if (c->world == 1) { memcpy(recv, send, bytes_per_rank); return KOMBGPU_OK; }
    const int rc = c->allgather(c->user, send, recv, (uint64_t)bytes_per_rank);
    return rc == 0 ? KOMBGPU_OK : KOMBGPU_ESTATE;
}

SymMark sym_mark(const kombgpu_comm *c) {
    // the allocation cursor is the last segment that holds anything
    size_t s = 0;
    for (size_t i = 0; i < c->segs.size(); ++i)
        if (c->segs[i].used) s = i;
    return SymMark{s, c->segs.empty() ? 0 : c->segs[s].used};
}

void sym_release(kombgpu_comm *c, SymMark m) {
    for (size_t i = 0; i < c->segs.size(); ++i) {
        if (i > m.seg) c->segs[i].used = 0;
        else if (i == m.seg) c->segs[i].used = m.used;
    }
}

int sym_alloc_bytes(kombgpu_comm *c, size_t bytes, void **local, void **peers) {
    bytes = (bytes + 511) & ~(size_t)511;
    // first segment at or after the cursor with room on top (identical on every rank: same call sequence, same sizes)
    const SymMark cur = sym_mark(c);
    size_t pick = c->segs.size();
    for (size_t i = cur.seg; i < c->segs.size(); ++i)
        if (c->segs[i].bytes - c->segs[i].used >= bytes) { pick = i; break; }
    if (pick == c->segs.size()) {
        const size_t want = bytes > c->seg_bytes ? bytes : c->seg_bytes;
        KG_TRY(new_segment(c, want));
    }
    SymSegment &s = c->segs[pick];
    *local = static_cast<char *>(s.local) + s.used;
    for (int q = 0; q < kMaxRanks; ++q) peers[q] = q < c->world ? static_cast<char *>(s.peer[q]) + s.used : nullptr;
    s.used += bytes;
    uint64_t total = 0;
    for (auto &g : c->segs) total += g.bytes;
    if (total > c->sym_high_water) c->sym_high_water = total;
    return KOMBGPU_OK;
}

int comm_exchange(kombgpu_comm *c, const unsigned long long *vals, int k, unsigned long long *out) {
    kombgpu_ctx *ctx = c->ctx;
    if (k < 1 || k > kCtlWords) return ctx_fail(ctx, KOMBGPU_EINVAL, "comm_exchange: %d words", k);
    if (c->world == 1) {
        KG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        memcpy(out, vals, (size_t)k * sizeof(unsigned long long));
        return KOMBGPU_OK;
    }
    if (!c->device_wait_ok) {
        // ranks share one device: a kernel must not wait for another rank's kernel.  The host threads meet instead.
        KG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        if (group_allgather(c, vals, out, (uint64_t)k * sizeof(unsigned long long)) != 0)
            return ctx_fail(ctx, KOMBGPU_ESTATE, "a rank of the local group failed");
        return KOMBGPU_OK;
    }
    ExchangeWords w{};
    for (int j = 0; j < k; ++j) w.w[j] = vals[j];
    const unsigned long long epoch = ++c->epoch;
    KG_LAUNCH(ctx, exchange_kernel, 1, 32, 0, c->ctl_peers, c->rank, c->world, epoch, w, k, c->xchg_out);
    KG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (c->xchg_out[c->world * k]) return ctx_fail(ctx, KOMBGPU_EINTERNAL, "exchange %llu: a peer rank did not arrive within 30 s", epoch);
    memcpy(out, c->xchg_out, (size_t)c->world * k * sizeof(unsigned long long));
    return KOMBGPU_OK;
}

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

int comm_group_barrier(kombgpu_comm *c) {
    if (!c->group) return KOMBGPU_OK;
    if (group_barrier(c->group) != KOMBGPU_OK) return ctx_fail(c->ctx, KOMBGPU_ESTATE, "a rank of the local group failed");
    return KOMBGPU_OK;
}

int comm_allreduce_sum(kombgpu_comm *c, unsigned long long v, unsigned long long *out) {
    unsigned long long all[kMaxRanks];
    KG_TRY(comm_exchange(c, &v, 1, all));
    unsigned long long s = 0;
    for (int q = 0; q < c->world; ++q) s += all[q];
    *out = s;
    return KOMBGPU_OK;
}

}  // namespace kg

using namespace kg;

static int comm_setup(kombgpu_comm *c, uint64_t heap_bytes) {
    kombgpu_ctx *ctx = c->ctx;
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    BootInfo mine{}, all[kMaxRanks];
    mine.pid = (int)getpid();
    mine.device = ctx->device;
    mine.in_group = c->group ? 1 : 0;
    mine.host_hash = hostname_hash();
    cudaDeviceGetPCIBusId(mine.bus_id, sizeof(mine.bus_id), ctx->device);
    if (comm_bootstrap_allgather(c, &mine, all, sizeof(BootInfo)) != KOMBGPU_OK)
        return ctx_fail(ctx, KOMBGPU_ESTATE, "communicator bootstrap all-gather failed");
    // topology: every rank on its own GPU of this host, or (tests) every rank on the same GPU of one process
    int distinct = 0, same_as_mine = 0;
    for (int q = 0; q < c->world; ++q) {
        if (all[q].host_hash != mine.host_hash)
            return ctx_fail(ctx, KOMBGPU_EINVAL, "rank %d runs on another host: the peer-memory path is single-node", q);
        if (strncmp(all[q].bus_id, mine.bus_id, sizeof(mine.bus_id)) == 0) ++same_as_mine;
        bool first = true;
        for (int r = 0; r < q; ++r) first = first && strncmp(all[r].bus_id, all[q].bus_id, sizeof(mine.bus_id)) != 0;
        distinct += first ? 1 : 0;
    }
    if (distinct == c->world) {
        c->same_device = false;
        c->device_wait_ok = true;
    } else if (distinct == 1 && c->group) {
        c->same_device = true;      // emulation: host-side exchange, one cooperative grid for the peel
        c->device_wait_ok = false;
    } else {
        return ctx_fail(ctx, KOMBGPU_EINVAL,
                        "%d ranks on %d GPUs: every rank needs its own GPU (ranks sharing a device would wait for one another "
                        "on it); only the ranks of one process may share one device (emulation for tests)", c->world, distinct);
    }
    if (!c->same_device) {
        for (int q = 0; q < c->world; ++q) {
            if (q == c->rank) continue;
            int can = 0;
            // between processes the ordinal of the peer is not ours to ask about: cudaIpcOpenMemHandle reports it
            if (c->group) {
                KG_CUDA(ctx, cudaDeviceCanAccessPeer(&can, ctx->device, all[q].device));
                if (!can) return ctx_fail(ctx, KOMBGPU_ENODEV, "device %d cannot access device %d (no peer path)", ctx->device, all[q].device);
                cudaError_t e = cudaDeviceEnablePeerAccess(all[q].device, 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled)
                    return ctx_fail(ctx, KOMBGPU_ECUDA, "cudaDeviceEnablePeerAccess(%d): %s", all[q].device, cudaGetErrorString(e));
                cudaGetLastError();
            }
        }
    }
    c->seg_bytes = heap_bytes ? (size_t)heap_bytes : ((size_t)512 << 20);
    // segment 0 starts with the control block
    CtlBlock *ctl = nullptr;
    KG_TRY(sym_alloc(c, 1, &ctl, &c->ctl_peers));
    c->ctl = ctl;
    if (cudaMallocHost(&c->xchg_out, (kMaxRanks * kCtlWords + 1) * sizeof(unsigned long long)) != cudaSuccess) {
        cudaGetLastError();
        return ctx_fail(ctx, KOMBGPU_ENOMEM, "pinned exchange buffer");
    }
    // everyone's control block is zeroed (new_segment) before anyone writes a flag
    int token = 1, tokens[kMaxRanks];
    if (comm_bootstrap_allgather(c, &token, tokens, sizeof(int)) != KOMBGPU_OK)
        return ctx_fail(ctx, KOMBGPU_ESTATE, "communicator bootstrap barrier failed");
    return KOMBGPU_OK;
}

static void comm_free(kombgpu_comm *c) {
    if (!c) return;
    if (c->ctx) {
        cudaSetDevice(c->ctx->device);
        cudaStreamSynchronize(c->ctx->stream);
    }
    for (auto &s : c->segs) {
        for (int q = 0; q < kMaxRanks; ++q)
            if (s.ipc_opened[q]) cudaIpcCloseMemHandle(s.peer[q]);
        if (s.local) cudaFree(s.local);
    }
    if (c->xchg_out) cudaFreeHost(c->xchg_out);
    if (c->group) {
        bool last;
        {
            std::lock_guard<std::mutex> lk(c->group->mu);
            last = --c->group->refs == 0;
        }
        if (last) delete c->group;
    }
    delete c;
}

extern "C" {

int kombgpu_comm_create(kombgpu_ctx *ctx, int rank, int world, kombgpu_allgather_fn allgather, void *user, uint64_t heap_bytes,
                        kombgpu_comm **out) {
    if (!ctx) return KOMBGPU_EINVAL;
    if (!out || world < 1 || world > kMaxRanks || rank < 0 || rank >= world || (world > 1 && !allgather))
        return ctx_fail(ctx, KOMBGPU_EINVAL, "kombgpu_comm_create: bad argument (1 <= world <= %d)", kMaxRanks);
    *out = nullptr;
    kombgpu_comm *c = new (std::nothrow) kombgpu_comm();
    if (!c) return ctx_fail(ctx, KOMBGPU_ENOMEM, "host allocation");
    c->ctx = ctx;
    c->rank = rank;
    c->world = world;
    c->allgather = allgather;
    c->user = user;
    const int rc = comm_setup(c, heap_bytes);
    if (rc != KOMBGPU_OK) { comm_free(c); return rc; }
    *out = c;
    return KOMBGPU_OK;
}

// The ranks of one process.  Call it from `world` host threads, one per rank, each with its own context; `group_key`
// (any address shared by the callers, e.g. the array of contexts) names the group.  Collective.
int kombgpu_comm_create_local(kombgpu_ctx *ctx, int rank, int world, void **group_slot, uint64_t heap_bytes, kombgpu_comm **out) {
    if (!ctx) return KOMBGPU_EINVAL;
    if (!out || !group_slot || world < 1 || world > kMaxRanks || rank < 0 || rank >= world)
        return ctx_fail(ctx, KOMBGPU_EINVAL, "kombgpu_comm_create_local: bad argument (1 <= world <= %d)", kMaxRanks);
    *out = nullptr;
    // the first caller creates the group object in *group_slot (the callers share the slot; it must start as NULL)
    static std::mutex slot_mu;
    LocalGroup *g;
    {
        std::lock_guard<std::mutex> lk(slot_mu);
        if (!*group_slot) {
            g = new (std::nothrow) LocalGroup();
            if (!g) return ctx_fail(ctx, KOMBGPU_ENOMEM, "host allocation");
            g->world = world;
            *group_slot = g;
        }
        g = static_cast<LocalGroup *>(*group_slot);
        if (g->world != world) return ctx_fail(ctx, KOMBGPU_EINVAL, "group was created for %d ranks, not %d", g->world, world);
        ++g->refs;
    }
    kombgpu_comm *c = new (std::nothrow) kombgpu_comm();
    if (!c) return ctx_fail(ctx, KOMBGPU_ENOMEM, "host allocation");
    c->ctx = ctx;
    c->rank = rank;
    c->world = world;
    c->group = g;
    c->allgather = group_allgather;
    c->user = c;
    const int rc = comm_setup(c, heap_bytes);
    if (rc != KOMBGPU_OK) {
        {   // the other ranks must not wait for this one for ever
            std::lock_guard<std::mutex> lk(g->mu);
            g->broken = true;
        }
        g->cv.notify_all();
        comm_free(c);
        return rc;
    }
    *out = c;
    return KOMBGPU_OK;
}

void kombgpu_comm_destroy(kombgpu_comm *c) { comm_free(c); }

// A rank of a local group that cannot go on (its host code failed) releases the ranks that wait for it.
int kombgpu_comm_abort(kombgpu_comm *c) {
    if (!c) return KOMBGPU_EINVAL;
    if (c->group) {
        {
            std::lock_guard<std::mutex> lk(c->group->mu);
            c->group->broken = true;
        }
        c->group->cv.notify_all();
    }
    return KOMBGPU_OK;
}

int kombgpu_comm_info(const kombgpu_comm *c, int *rank, int *world, int *same_device, uint64_t *heap_bytes) {
    if (!c) return KOMBGPU_EINVAL;
    if (rank) *rank = c->rank;
    if (world) *world = c->world;
    if (same_device) *same_device = c->same_device ? 1 : 0;
    if (heap_bytes) *heap_bytes = c->sym_high_water;
    return KOMBGPU_OK;
}

}  // extern "C"
