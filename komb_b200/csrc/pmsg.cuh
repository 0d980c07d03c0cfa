// pmsg.cuh — what the text stages over the ranks of a communicator share (psam.cu, pfasta.cu): byte slices of a host
// file that never split a line, status words gathered over the ranks, and a sender of variable-length strings.  send_msgs
// scans the sizes once per destination and stores every message and its bytes into the destination's receive buffers
// (symmetric heap, peer memory), sized by an exchanged count matrix as in route_keys.  Replies are single stores into
// the sender's reply array at the index the message carries; the caller's kernels make them.
#pragma once

#include <cstring>
#include <vector>

#include "comm.cuh"
#include "primitives.cuh"
#include "strings.cuh"

namespace kg {
namespace {

struct Msg {             // one item sent to a rank
    uint64_t key;        // the sender's payload (psam.cu: the occurrence key of a name)
    uint64_t off;        // where its bytes start in the receiver's byte buffer
    uint32_t len;        // length of its string
    uint32_t idx;        // the sender's index of the item: where a reply goes
    uint32_t rank;       // the sender
    uint32_t flag;       // the name has a hit on the sender
};

struct Inbox {
    Msg *msg = nullptr;
    unsigned char *bytes = nullptr;
    uint64_t n = 0, n_bytes = 0;
};

struct DestFlagIn {
    const uint32_t *dest;
    uint32_t d;
    __device__ uint32_t operator()(uint64_t i) const { return dest[i] == d ? 1u : 0u; }
};
struct DestSlotOut {
    uint32_t *slot;
    __device__ void operator()(uint64_t i, uint32_t prefix, uint32_t flag) const {
        if (flag) slot[i] = prefix;
    }
};
struct DestBytesIn {
    const uint32_t *dest;
    const Msg *msg;
    uint32_t d;
    __device__ uint64_t operator()(uint64_t i) const { return dest[i] == d ? (uint64_t)msg[i].len : 0ull; }
};
struct DestBytesOut {
    const uint32_t *dest;
    uint32_t d;
    uint64_t *boff;
    __device__ void operator()(uint64_t i, uint64_t prefix, uint64_t) const {
        if (dest[i] == d) boff[i] = prefix;
    }
};

struct SendBase {   // where this rank's run starts in every destination's buffers
    unsigned long long slot[kMaxRanks], byte[kMaxRanks];
};

// one warp per message: lane 0 stores the message, the lanes store its bytes
__global__ void __launch_bounds__(kThreads) send_kernel(const Msg *__restrict__ msg, const uint32_t *__restrict__ dest,
                                                        const uint32_t *__restrict__ slot, const uint64_t *__restrict__ boff,
                                                        const unsigned char *__restrict__ text, const uint64_t *__restrict__ src_off, uint64_t n,
                                                        SendBase base, PeerPtrs<Msg> dmsg, PeerPtrs<unsigned char> dbytes) {
    const uint64_t warps = (uint64_t)gridDim.x * (blockDim.x >> 5);
    for (uint64_t i = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n; i += warps) {
        const uint32_t d = dest[i];
        Msg m = msg[i];
        if (src_off) {
            m.off = base.byte[d] + boff[i];
            const unsigned char *s = text + src_off[i];
            unsigned char *t = dbytes.p[d] + m.off;
            for (uint32_t k = lane_id(); k < m.len; k += 32) t[k] = s[k];
        }
        if (lane_id() == 0) dmsg.p[d][base.slot[d] + slot[i]] = m;
    }
}

// All-gather of mine.size() words per rank (any number: exchanges of kCtlWords words each).  Word 0 is the rank's
// status: when a rank has failed, every rank returns an error (the failing rank its own; the others name `stage`).
int gather_words(kombgpu_comm *c, int rc_local, std::vector<unsigned long long> &mine, std::vector<unsigned long long> &all,
                 const char *stage) {
    const int k = (int)mine.size(), world = c->world;
    mine[0] = rc_local != KOMBGPU_OK ? (unsigned long long)-rc_local : 0ull;
    all.assign((size_t)world * k, 0ull);
    unsigned long long part[kMaxRanks * kCtlWords];
    for (int j0 = 0; j0 < k; j0 += kCtlWords) {
        const int kk = k - j0 < kCtlWords ? k - j0 : kCtlWords;
        KG_TRY(comm_exchange(c, mine.data() + j0, kk, part));
        for (int q = 0; q < world; ++q)
            for (int j = 0; j < kk; ++j) all[(size_t)q * k + j0 + j] = part[q * kk + j];
    }
    if (rc_local != KOMBGPU_OK) return rc_local;
    for (int q = 0; q < world; ++q)
        if (all[(size_t)q * k]) return ctx_fail(c->ctx, -(int)all[(size_t)q * k], "rank %d failed; %s stopped on every rank", q, stage);
    return KOMBGPU_OK;
}

int barrier(kombgpu_comm *c, int rc_local, const char *stage) {
    std::vector<unsigned long long> mine(1), all;
    return gather_words(c, rc_local, mine, all, stage);
}

// Collective: message i (and, with src_off, the string text[src_off[i] .. + len)) goes to rank dest[i].  The messages
// a rank receives arrive in sender order, each sender's in its own order; they live in the symmetric heap.
int send_msgs(kombgpu_comm *c, int rc, const Msg *msg, const uint32_t *dest, uint64_t n, const unsigned char *text, const uint64_t *src_off,
              Inbox *in, const char *stage) {
    kombgpu_ctx *ctx = c->ctx;
    const int world = c->world, rank = c->rank;
    std::vector<unsigned long long> mine(1 + 2 * (size_t)world, 0ull), all;
    DevBuf<uint32_t> slot, d_cnt;
    DevBuf<uint64_t> boff, d_bytes;
    if (rc == KOMBGPU_OK) rc = [&]() -> int {
        KG_ALLOC(ctx, slot, n);
        KG_ALLOC(ctx, boff, n);
        KG_ALLOC(ctx, d_cnt, world);
        KG_ALLOC(ctx, d_bytes, world);
        for (int d = 0; d < world; ++d) {   // one size scan per destination: the messages' slots, the strings' offsets
            KG_TRY((device_scan<uint32_t>(ctx, n, DestFlagIn{dest, (uint32_t)d}, DestSlotOut{slot.p}, d_cnt.p + d)));
            if (src_off) KG_TRY((device_scan<uint64_t>(ctx, n, DestBytesIn{dest, msg, (uint32_t)d}, DestBytesOut{dest, (uint32_t)d, boff.p}, d_bytes.p + d)));
        }
        std::vector<uint32_t> cnt(world);
        std::vector<uint64_t> bytes(world, 0);
        KG_TRY(read_back(ctx, d_cnt.p, cnt.data(), world));
        if (src_off) KG_TRY(read_back(ctx, d_bytes.p, bytes.data(), world));
        for (int d = 0; d < world; ++d) { mine[1 + d] = cnt[d]; mine[1 + world + d] = bytes[d]; }
        return KOMBGPU_OK;
    }();
    KG_TRY(gather_words(c, rc, mine, all, stage));
    SendBase base{};
    unsigned long long max_n = 0, max_bytes = 0;
    for (int p = 0; p < world; ++p) {
        unsigned long long nt = 0, bt = 0;
        for (int q = 0; q < world; ++q) {
            if (q == rank) { base.slot[p] = nt; base.byte[p] = bt; }
            nt += all[(size_t)q * (1 + 2 * world) + 1 + p];
            bt += all[(size_t)q * (1 + 2 * world) + 1 + world + p];
        }
        if (p == rank) { in->n = nt; in->n_bytes = bt; }
        max_n = nt > max_n ? nt : max_n;
        max_bytes = bt > max_bytes ? bt : max_bytes;
    }
    if (max_n >= 0xffffffffull) return ctx_fail(ctx, KOMBGPU_EINVAL, "%llu strings sent to one rank exceed its 2^32 - 1 limit", max_n);
    PeerPtrs<Msg> pmsg{};
    PeerPtrs<unsigned char> pbytes{};
    KG_TRY(sym_alloc(c, (size_t)max_n, &in->msg, &pmsg));
    KG_TRY(sym_alloc(c, (size_t)max_bytes, &in->bytes, &pbytes));
    if (n) rc = [&]() -> int {
        KG_LAUNCH(ctx, send_kernel, grid_for(n * 32, kThreads, ctx->sm_count), kThreads, 0, msg, dest, slot.p, boff.p, text, src_off, n, base,
                  pmsg, pbytes);
        return KOMBGPU_OK;
    }();
    return barrier(c, rc, stage);   // everything every rank stored has landed
}

// cut[q * n_files + f] = the first line start at or after floor(size_f * q / world) -- with lead != 0, the first line
// start that holds the byte `lead` (a FASTA record: '>'); cut[f] = 0 and cut[world * n_files + f] = size_f
void slice_cuts(const char *const *texts, const uint64_t *sizes, int n_files, int world, char lead, std::vector<uint64_t> &cut) {
    cut.assign((size_t)(world + 1) * n_files, 0);
    const char pat[2] = {'\n', lead};
    for (int f = 0; f < n_files; ++f)
        for (int q = 1; q <= world; ++q) {
            const char *t = texts[f];
            const uint64_t size = sizes[f];
            uint64_t x = q == world ? size : (uint64_t)((unsigned __int128)size * (unsigned)q / (unsigned)world);
            if (lead && x < size && !(t[x] == lead && (x == 0 || t[x - 1] == '\n'))) {
                const uint64_t from = x ? x - 1 : 0;
                const void *p = memmem(t + from, size - from, pat, 2);
                x = p ? (uint64_t)(static_cast<const char *>(p) - t) + 1 : size;
            } else if (!lead && x > 0 && x < size && t[x - 1] != '\n') {
                const void *nl = memchr(t + x, '\n', size - x);
                x = nl ? (uint64_t)(static_cast<const char *>(nl) - t) + 1 : size;
            }
            cut[(size_t)q * n_files + f] = x;
        }
}

}  // namespace
}  // namespace kg
