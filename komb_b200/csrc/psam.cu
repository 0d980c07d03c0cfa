// psam.cu — SAM text -> hits over the ranks of a communicator (kombgpu_dist_sam_parse, DESIGN.md §4 "SAM text over
// the ranks").  Same token rules, unitig numbering and error messages as sam.cu, whose kernels (sam.cuh) do the work
// inside a rank:
//   1. local parse   rank q uploads the lines that start in its byte slice of every input, counts their newlines,
//                    parses, compacts and interns its read keys and names locally.  The ranks exchange their line
//                    counts per input and their earliest malformed line: global line numbers, one agreed error
//   2. read keys     every distinct local key goes (length + bytes) to its OWNER, the rank a fixed-seed hash of its
//                    bytes picks; the owner interns what it received by the bytes (intern_items) and stores each key's
//                    id, owner * stride + local id, into the sender's reply slot
//   3. unitig names  the same for the distinct local names, each with the key of its first occurrence on the sender
//                    (class: @SQ 0 / hit 1, input, byte offset inside the input) and whether it has a hit there; the
//                    owner keeps the smallest key and ORs the flags
//   4. vids          the owner sends the smallest key of every name with a hit to the key's HOME, the rank whose slice
//                    holds that byte.  A home sorts the keys it received; the ranks exchange their counts per (class,
//                    input), so vid = global offset of the group + offset of the home in it + rank in the home's sort.
//                    The vid goes back home -> owner -> sender; the home also stores (input, offset, length) of the
//                    vid in the rank that owns the vid's range (kombgpu_dist_hits_names), and sends it the name's
//                    bytes, which it still holds: the owner formats kcore.tsv rows from them (format.cu)
//   5. routing       (read id << 32 | vid) of every hit goes to the owner of its read: route_keys (pbuild.cu)
// Steps 2-4 send variable-length strings, which route_keys (fixed 64-bit keys) cannot carry: send_msgs (pmsg.cuh)
// scans the sizes once per destination and stores every message and its bytes into the destination's receive buffers
// (symmetric heap, peer memory), sized by an exchanged count matrix as in route_keys.  A reply is one store into the
// sender's reply array at the index the message carries.
#include <cstring>
#include <new>
#include <vector>

#include "dgraph.cuh"
#include "pmsg.cuh"
#include "sam.cuh"

struct kombgpu_dist_hits {
    kombgpu_comm *comm = nullptr;
    kombgpu_ctx *ctx = nullptr;
    uint64_t n_hits_local = 0, n_hits_global = 0, n_lines_global = 0;
    uint32_t n_reads_global = 0, n_unitigs = 0, v_lo = 0, n_local = 0;
    uint32_t *read_key = nullptr;   // [n_hits_local] routed hits
    uint32_t *unitig = nullptr;     // [n_hits_local]
    uint64_t *name_key = nullptr;   // [n_local] input << 56 | offset inside that input, of vertex v_lo + i
    uint32_t *name_len = nullptr;   // [n_local]
    unsigned char *name_bytes = nullptr;   // the bytes of the names of vertices [v_lo, v_lo + n_local), in no order
    uint64_t *name_off = nullptr;          // [n_local] where the name of vertex v_lo + i starts in name_bytes
    float ms_upload = 0.f, ms_parse = 0.f, ms_intern = 0.f, ms_route = 0.f;
    int hash_rounds = 0;
};

namespace kg {
namespace {

constexpr uint64_t kOwnerSeed = 0x2545f4914f6cdd1dull;   // picks a string's owner: the same on every rank, never changed
constexpr int kKeyFileShift = 56;                        // occurrence key: class << 63 | input << 56 | offset
constexpr uint64_t kKeyOffMask = (1ull << kKeyFileShift) - 1;
constexpr uint64_t kKeyClassHit = 1ull << 63;
constexpr const char *kStage = "the SAM parse";   // named in the error of a rank whose peer failed

// the received strings as items to intern
__global__ void __launch_bounds__(kThreads) inbox_items_kernel(const Msg *__restrict__ msg, uint64_t n, const unsigned char *__restrict__ bytes,
                                                               uint64_t seed, Items out) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const Msg m = msg[i];
        out.off[i] = m.off;
        out.len[i] = m.len;
        out.hash[i] = hash_span(bytes + m.off, m.len, seed);
    }
}

// distinct local key k (its first item) -> message to the key's owner
__global__ void __launch_bounds__(kThreads) key_msgs_kernel(const unsigned char *__restrict__ text, Items keys, const uint32_t *__restrict__ first,
                                                            uint64_t n, int world, int rank, Msg *__restrict__ msg, uint32_t *__restrict__ dest,
                                                            uint64_t *__restrict__ src_off) {
    for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t f = first[k];
        const uint64_t off = keys.off[f];
        const uint32_t len = keys.len[f];
        dest[k] = (uint32_t)(hash_span(text + off, len, kOwnerSeed) % (uint64_t)world);
        msg[k] = Msg{0ull, 0ull, len, (uint32_t)k, (uint32_t)rank, 0u};
        src_off[k] = off;
    }
}

struct Slices {   // this rank's slices in its text buffer
    const uint64_t *base;     // [n_files] offset of slice f in the buffer
    const uint64_t *cut_lo;   // [n_files] offset of slice f in input f
    int n_files;
};

// distinct local name d (its first item: @SQ records come first) -> message to the name's owner, with the key of
// its first occurrence here and whether it has a hit here
__global__ void __launch_bounds__(kThreads) name_msgs_kernel(const unsigned char *__restrict__ text, Items items, const uint32_t *__restrict__ first,
                                                             uint64_t n, uint64_t n_sq, const uint32_t *__restrict__ used, Slices sl, int world,
                                                             int rank, Msg *__restrict__ msg, uint32_t *__restrict__ dest, uint64_t *__restrict__ src_off) {
    for (uint64_t d = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; d < n; d += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t fi = first[d];
        const uint64_t off = items.off[fi];
        const uint32_t len = items.len[fi];
        int f = 0;   // the last slice that starts at or before the name (empty slices before it start at the same byte)
        for (int g = 1; g < sl.n_files; ++g)
            if (sl.base[g] <= off) f = g;
        const uint64_t key = (fi < n_sq ? 0ull : kKeyClassHit) | ((uint64_t)f << kKeyFileShift) | (off - sl.base[f] + sl.cut_lo[f]);
        dest[d] = (uint32_t)(hash_span(text + off, len, kOwnerSeed) % (uint64_t)world);
        msg[d] = Msg{key, 0ull, len, (uint32_t)d, (uint32_t)rank, used[d]};
        src_off[d] = off;
    }
}

// owner: the global id of every received key goes into its sender's reply slot
__global__ void __launch_bounds__(kThreads) reply_kernel(const Msg *__restrict__ msg, uint64_t n, const uint32_t *__restrict__ ids, uint32_t id_base,
                                                         PeerPtrs<uint32_t> reply) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const Msg m = msg[i];
        reply.p[m.rank][m.idx] = id_base + ids[i];
    }
}

// owner: smallest occurrence key and OR of the hit flags of every distinct name
__global__ void __launch_bounds__(kThreads) name_merge_kernel(const Msg *__restrict__ msg, uint64_t n, const uint32_t *__restrict__ ids,
                                                              unsigned long long *__restrict__ min_key, uint32_t *__restrict__ hit,
                                                              uint32_t *__restrict__ len) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const Msg m = msg[i];
        const uint32_t d = ids[i];
        atomicMin(&min_key[d], (unsigned long long)m.key);
        if (m.flag) atomicOr(&hit[d], 1u);
        len[d] = m.len;   // equal names, equal lengths
    }
}

__device__ __forceinline__ uint32_t key_home(uint64_t key, const uint64_t *__restrict__ cut, int n_files, int world) {
    const int f = (int)((key >> kKeyFileShift) & 63u);
    const uint64_t off = key & kKeyOffMask;
    uint32_t q = 0;   // the last slice that starts at or before the byte (empty slices start where the next one does)
    for (int r = 1; r < world; ++r)
        if (cut[(size_t)r * n_files + f] <= off) q = (uint32_t)r;
    return q;
}

struct HitNameOut {   // owner: a distinct name with a hit -> message to the home of its first occurrence
    const unsigned long long *min_key;
    const uint32_t *len;
    const uint64_t *cut;
    int n_files, world, rank;
    Msg *msg;
    uint32_t *dest;
    __device__ void operator()(uint64_t d, uint32_t p, uint32_t flag) const {
        if (!flag) return;
        msg[p] = Msg{min_key[d], 0ull, len[d], (uint32_t)d, (uint32_t)rank, 1u};
        dest[p] = key_home(min_key[d], cut, n_files, world);
    }
};

__global__ void __launch_bounds__(kThreads) msg_keys_kernel(const Msg *__restrict__ msg, uint64_t n, int n_files, uint64_t *__restrict__ keys,
                                                            unsigned long long *__restrict__ group_cnt) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t k = msg[i].key;
        keys[i] = k;
        atomicAdd(&group_cnt[(k >> 63) * n_files + ((k >> kKeyFileShift) & 63u)], 1ull);
    }
}

// home: vid = rank of the key among the home's sorted keys + the offset of its (class, input) group; the vid goes to
// the owner of the name, the name's span to the owner of the vid.  out / dest / src_off: the message that carries the
// name's bytes (in this rank's text buffer) to the owner of the vid, idx = vid - owner * step
__global__ void __launch_bounds__(kThreads) vid_kernel(const Msg *__restrict__ msg, uint64_t n, const uint64_t *__restrict__ sorted,
                                                       const unsigned long long *__restrict__ delta, int n_files, uint32_t step,
                                                       PeerPtrs<uint32_t> vid_reply, PeerPtrs<uint64_t> name_key, PeerPtrs<uint32_t> name_len,
                                                       Slices sl, Msg *__restrict__ out, uint32_t *__restrict__ dest, uint64_t *__restrict__ src_off) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const Msg m = msg[i];
        uint64_t lo = 0, hi = n;   // the keys are distinct: lower bound = rank
        while (lo < hi) {
            const uint64_t mid = (lo + hi) >> 1;
            if (sorted[mid] < m.key) lo = mid + 1;
            else hi = mid;
        }
        const uint32_t vid = (uint32_t)(lo + delta[(m.key >> 63) * n_files + ((m.key >> kKeyFileShift) & 63u)]);
        vid_reply.p[m.rank][m.idx] = vid;
        const uint32_t o = vid / step;
        name_key.p[o][vid - o * step] = m.key & ~kKeyClassHit;
        name_len.p[o][vid - o * step] = m.len;
        const uint32_t f = (uint32_t)((m.key >> kKeyFileShift) & 63u);
        out[i] = Msg{0ull, 0ull, m.len, vid - o * step, 0u, 0u};
        dest[i] = o;
        src_off[i] = sl.base[f] + (m.key & kKeyOffMask) - sl.cut_lo[f];
    }
}

// owner: where the name of each of its vertices starts in the received bytes
__global__ void __launch_bounds__(kThreads) name_off_kernel(const Msg *__restrict__ msg, uint64_t n, uint64_t *__restrict__ name_off) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) name_off[msg[i].idx] = msg[i].off;
}

// owner: the vid of every received name goes into its sender's reply slot
__global__ void __launch_bounds__(kThreads) name_reply_kernel(const Msg *__restrict__ msg, uint64_t n, const uint32_t *__restrict__ ids,
                                                              const uint32_t *__restrict__ vid, PeerPtrs<uint32_t> reply) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const Msg m = msg[i];
        reply.p[m.rank][m.idx] = vid[ids[i]];
    }
}

// (read id << 32 | vid) of every local hit
__global__ void __launch_bounds__(kThreads) hit_keys_kernel(const uint32_t *__restrict__ key_ids, const uint32_t *__restrict__ read_id,
                                                            const uint32_t *__restrict__ name_ids, const uint32_t *__restrict__ vid, uint64_t n,
                                                            uint64_t *__restrict__ out) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
        out[i] = ((uint64_t)read_id[key_ids[i]] << 32) | vid[name_ids[i]];
}

__global__ void __launch_bounds__(kThreads) split_hits_kernel(const uint64_t *__restrict__ keys, uint64_t n, uint32_t *__restrict__ read_key,
                                                              uint32_t *__restrict__ unitig) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        read_key[i] = (uint32_t)(keys[i] >> 32);
        unitig[i] = (uint32_t)keys[i];
    }
}

int dist_sam_parse(kombgpu_comm *c, const char *const *texts, const uint64_t *sizes, int n_files, kombgpu_dist_hits *h) {
    kombgpu_ctx *ctx = c->ctx;
    const int world = c->world, rank = c->rank, F = n_files;
    SymRewind heap{c, sym_mark(c)};
    EvTimer tm(ctx);
    std::vector<uint64_t> cut;
    slice_cuts(texts, sizes, F, world, 0, cut);
    std::vector<uint64_t> base(F, 0), cut_lo(F), len(F);
    uint64_t total = 0;
    for (int f = 0; f < F; ++f) {
        cut_lo[f] = cut[(size_t)rank * F + f];
        len[f] = cut[(size_t)(rank + 1) * F + f] - cut_lo[f];
        base[f] = total;
        total += (len[f] + 15) & ~15ull;
    }

    // ---- 1. upload this rank's slices, count and parse their lines
    DevBuf<unsigned char> text;
    DevBuf<unsigned long long> d_cnt;   // [error word | newlines per slice]
    DevBuf<uint64_t> d_cut, d_base, d_cut_lo;
    std::vector<unsigned long long> n_lines((size_t)F + 1, 0);
    std::vector<uint64_t> line_base(F, 0);
    uint64_t nl = 0;
    int rc = [&]() -> int {
        KG_ALLOC(ctx, text, total ? total : 16);
        for (int f = 0; f < F; ++f) {
            if (len[f]) KG_CUDA(ctx, cudaMemcpyAsync(text.p + base[f], texts[f] + cut_lo[f], len[f], cudaMemcpyHostToDevice, ctx->stream));
            const uint64_t pad = ((len[f] + 15) & ~15ull) - len[f];
            if (pad) KG_CUDA(ctx, cudaMemsetAsync(text.p + base[f] + len[f], 0, pad, ctx->stream));
        }
        h->ms_upload = tm.lap();
        KG_ALLOC(ctx, d_cnt, (size_t)F + 1);
        KG_CUDA(ctx, cudaMemsetAsync(d_cnt.p, 0xff, sizeof(unsigned long long), ctx->stream));
        KG_CUDA(ctx, cudaMemsetAsync(d_cnt.p + 1, 0, (size_t)F * sizeof(unsigned long long), ctx->stream));
        for (int f = 0; f < F; ++f) {
            const uint64_t chunks = (len[f] + 15) / 16;
            if (chunks)
                KG_LAUNCH(ctx, newline_count_kernel, grid_for(chunks, kThreads * 4, ctx->sm_count), kThreads, 0,
                          reinterpret_cast<const uint4 *>(text.p + base[f]), chunks, d_cnt.p + 1 + f);
        }
        KG_TRY(read_back(ctx, d_cnt.p, n_lines.data(), (size_t)F + 1));
        for (int f = 0; f < F; ++f) { line_base[f] = nl; nl += n_lines[f + 1]; }
        // sam.cu's per-call limit (its compaction scan packs two counters), applied to each rank's slices
        if (nl >= (1ull << 30)) return ctx_fail(ctx, KOMBGPU_EINVAL, "%llu lines in rank %d's slices exceed the 2^30 per-rank limit", (unsigned long long)nl, rank);
        KG_ALLOC(ctx, d_cut, cut.size());
        KG_ALLOC(ctx, d_base, F);
        KG_ALLOC(ctx, d_cut_lo, F);
        if (F) {
            KG_CUDA(ctx, cudaMemcpyAsync(d_cut.p, cut.data(), cut.size() * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream));
            KG_CUDA(ctx, cudaMemcpyAsync(d_base.p, base.data(), F * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream));
            KG_CUDA(ctx, cudaMemcpyAsync(d_cut_lo.p, cut_lo.data(), F * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream));
        }
        return KOMBGPU_OK;
    }();
    DevBuf<uint8_t> kind;
    ItemBufs lkey, lname, keys, rnames, sq;
    uint64_t n_hits = 0, n_sq = 0;
    unsigned long long h_err = ~0ull;
    uint64_t seed = 0x9e3779b97f4a7c15ull;
    if (rc == KOMBGPU_OK) rc = [&]() -> int {
        KG_ALLOC(ctx, kind, nl);
        KG_TRY(lkey.alloc(ctx, nl));
        KG_TRY(lname.alloc(ctx, nl));
        LineTable table{kind.p, lkey.off.p, lname.off.p, lkey.hash.p, lname.hash.p, lkey.len.p, lname.len.p};
        for (int f = 0; f < F; ++f) {
            const uint64_t L = n_lines[f + 1];
            if (!L) continue;
            DevBuf<uint64_t> start;
            KG_ALLOC(ctx, start, L + 1);
            KG_CUDA(ctx, cudaMemcpyAsync(start.p, &base[f], sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream));
            const uint4 *t4 = reinterpret_cast<const uint4 *>(text.p + base[f]);
            KG_TRY((device_scan<uint64_t>(ctx, (len[f] + 15) / 16, NewlineIn{t4}, LineStartOut{t4, base[f], start.p}, (uint64_t *)nullptr)));
            KG_LAUNCH(ctx, parse_lines_kernel, grid_for(L, kThreads, ctx->sm_count), kThreads, 0, text.p, start.p, L, line_base[f], seed, table,
                      d_cnt.p);
        }
        return read_back(ctx, d_cnt.p, &h_err, 1);
    }();
    // the ranks agree on the line numbers and on the earliest malformed line in (input, line) order
    {
        std::vector<unsigned long long> mine(2 + (size_t)F, 0ull), all;
        if (h_err != ~0ull) {
            const uint64_t line = h_err >> 2;
            int f = 0;
            while (f + 1 < F && line >= line_base[f + 1]) ++f;
            mine[1] = ((unsigned long long)f << 34) | ((line - line_base[f]) << 2) | (h_err & 3);
        } else {
            mine[1] = ~0ull;
        }
        for (int f = 0; f < F; ++f) mine[2 + f] = n_lines[f + 1];
        KG_TRY(gather_words(c, rc, mine, all, kStage));
        const size_t k = 2 + (size_t)F;
        int best_q = -1;
        for (int q = 0; q < world; ++q) {   // (input, rank, line) order = (input, line) order
            const unsigned long long e = all[q * k + 1];
            if (e == ~0ull) continue;
            const unsigned long long b = best_q < 0 ? ~0ull : all[best_q * k + 1];
            if (best_q < 0 || (e >> 34) < (b >> 34)) best_q = q;
        }
        h->n_lines_global = 0;
        for (int q = 0; q < world; ++q)
            for (int f = 0; f < F; ++f) h->n_lines_global += all[q * k + 2 + f];
        if (best_q >= 0) {
            const unsigned long long e = all[best_q * k + 1];
            const int f = (int)(e >> 34);
            unsigned long long line = ((e >> 2) & ((1ull << 32) - 1)) + 1;
            for (int q = 0; q < best_q; ++q) line += all[q * k + 2 + f];
            return ctx_fail(ctx, KOMBGPU_EINVAL, "malformed SAM (input %d, line %llu): %s", f, line,
                            (e & 3) == 1 ? "empty line" : "line with fewer than 3 tab-separated fields");
        }
    }
    // hits and @SQ records in file order, then the local interning
    DevBuf<uint32_t> key_ids, key_first, name_ids, name_first, used;
    ItemBufs items;
    uint32_t n_kd = 0, n_nd = 0;
    rc = [&]() -> int {
        DevBuf<uint64_t> d_tot(ctx, 1);
        if (!d_tot) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
        KG_TRY(keys.alloc(ctx, nl));
        KG_TRY(rnames.alloc(ctx, nl));
        KG_TRY(sq.alloc(ctx, nl));
        KG_TRY((device_scan<uint64_t>(ctx, nl, KindIn{kind.p}, CompactLines{LineTable{kind.p, lkey.off.p, lname.off.p, lkey.hash.p, lname.hash.p,
                                                                                      lkey.len.p, lname.len.p},
                                                                            keys.view(), rnames.view(), sq.view()},
                                      d_tot.p)));
        uint64_t tot = 0;
        KG_TRY(read_back(ctx, d_tot.p, &tot, 1));
        n_hits = tot & 0xffffffffull;
        n_sq = tot >> 32;
        kind.release();
        lkey.off.release(); lkey.hash.release(); lkey.len.release();
        lname.off.release(); lname.hash.release(); lname.len.release();
        h->ms_parse = tm.lap();
        KG_TRY(intern_items(ctx, text.p, keys.view(), n_hits, &seed, &h->hash_rounds, key_ids, key_first, &n_kd));
        const uint64_t n_items = n_sq + n_hits;
        KG_TRY(items.alloc(ctx, n_items));
        if (n_items)
            KG_LAUNCH(ctx, concat_items_kernel, grid_for(n_items, kThreads, ctx->sm_count), kThreads, 0, sq.view(), n_sq, rnames.view(), n_hits,
                      items.view());
        KG_TRY(intern_items(ctx, text.p, items.view(), n_items, &seed, &h->hash_rounds, name_ids, name_first, &n_nd));
        KG_ALLOC(ctx, used, n_nd);
        KG_CUDA(ctx, cudaMemsetAsync(used.p, 0, (size_t)(n_nd ? n_nd : 1) * sizeof(uint32_t), ctx->stream));
        if (n_hits) KG_LAUNCH(ctx, mark_used_kernel, grid_for(n_hits, kThreads, ctx->sm_count), kThreads, 0, name_ids.p + n_sq, n_hits, used.p);
        return KOMBGPU_OK;
    }();

    // ---- 2. read keys -> their owners, global ids back
    DevBuf<Msg> out_msg;
    DevBuf<uint32_t> out_dest;
    DevBuf<uint64_t> out_off;
    auto outbox = [&](uint64_t n) -> int {
        KG_ALLOC(ctx, out_msg, n);
        KG_ALLOC(ctx, out_dest, n);
        KG_ALLOC(ctx, out_off, n);
        return KOMBGPU_OK;
    };
    if (rc == KOMBGPU_OK) rc = [&]() -> int {
        KG_TRY(outbox(n_kd));
        if (n_kd)
            KG_LAUNCH(ctx, key_msgs_kernel, grid_for(n_kd, kThreads, ctx->sm_count), kThreads, 0, text.p, keys.view(), key_first.p, (uint64_t)n_kd,
                      world, rank, out_msg.p, out_dest.p, out_off.p);
        return KOMBGPU_OK;
    }();
    Inbox kin;
    KG_TRY(send_msgs(c, rc, out_msg.p, out_dest.p, n_kd, text.p, out_off.p, &kin, kStage));
    DevBuf<uint32_t> kin_ids, kin_first;
    uint32_t n_owned_keys = 0;
    rc = [&]() -> int {
        ItemBufs it;
        KG_TRY(it.alloc(ctx, kin.n));
        uint64_t s = 0x9e3779b97f4a7c15ull;
        if (kin.n) KG_LAUNCH(ctx, inbox_items_kernel, grid_for(kin.n, kThreads, ctx->sm_count), kThreads, 0, kin.msg, kin.n, kin.bytes, s, it.view());
        return intern_items(ctx, kin.bytes, it.view(), kin.n, &s, &h->hash_rounds, kin_ids, kin_first, &n_owned_keys);
    }();
    uint32_t stride = 1, max_nd = 1;
    uint32_t *read_id = nullptr;   // [distinct local key] its global id (symmetric heap, until the end)
    {
        std::vector<unsigned long long> mine = {0ull, n_owned_keys, n_kd, n_nd}, all;
        KG_TRY(gather_words(c, rc, mine, all, kStage));
        unsigned long long max_keys = 1, max_kd = 1, sum = 0;
        for (int q = 0; q < world; ++q) {
            max_keys = all[q * 4 + 1] > max_keys ? all[q * 4 + 1] : max_keys;
            max_kd = all[q * 4 + 2] > max_kd ? all[q * 4 + 2] : max_kd;
            max_nd = all[q * 4 + 3] > max_nd ? (uint32_t)all[q * 4 + 3] : max_nd;
            sum += all[q * 4 + 1];
        }
        if (max_keys * (unsigned long long)world > 0xffffffffull)
            return ctx_fail(ctx, KOMBGPU_EINVAL, "read ids (%llu distinct keys on one rank x %d ranks) exceed 32 bits", max_keys, world);
        stride = (uint32_t)max_keys;
        h->n_reads_global = (uint32_t)sum;
        PeerPtrs<uint32_t> preply{};
        KG_TRY(sym_alloc(c, (size_t)max_kd, &read_id, &preply));
        rc = [&]() -> int {
            if (kin.n) KG_LAUNCH(ctx, reply_kernel, grid_for(kin.n, kThreads, ctx->sm_count), kThreads, 0, kin.msg, kin.n, kin_ids.p, (uint32_t)rank * stride, preply);
            return KOMBGPU_OK;
        }();
        KG_TRY(barrier(c, rc, kStage));
        kin_ids.release();
        kin_first.release();
        key_first.release();
        keys.off.release(); keys.hash.release(); keys.len.release();
    }

    // ---- 3. unitig names -> their owners: smallest occurrence key, hit flag
    rc = [&]() -> int {
        KG_TRY(outbox(n_nd));
        if (n_nd)
            KG_LAUNCH(ctx, name_msgs_kernel, grid_for(n_nd, kThreads, ctx->sm_count), kThreads, 0, text.p, items.view(), name_first.p, (uint64_t)n_nd,
                      n_sq, used.p, Slices{d_base.p, d_cut_lo.p, F}, world, rank, out_msg.p, out_dest.p, out_off.p);
        return KOMBGPU_OK;
    }();
    Inbox nin;
    KG_TRY(send_msgs(c, rc, out_msg.p, out_dest.p, n_nd, text.p, out_off.p, &nin, kStage));
    DevBuf<uint32_t> nin_ids, nin_first, nhit, nlen;
    DevBuf<unsigned long long> nmin;
    uint32_t n_owned_names = 0, n_hit_names = 0;
    rc = [&]() -> int {
        ItemBufs it;
        KG_TRY(it.alloc(ctx, nin.n));
        uint64_t s = 0x9e3779b97f4a7c15ull;
        if (nin.n) KG_LAUNCH(ctx, inbox_items_kernel, grid_for(nin.n, kThreads, ctx->sm_count), kThreads, 0, nin.msg, nin.n, nin.bytes, s, it.view());
        KG_TRY(intern_items(ctx, nin.bytes, it.view(), nin.n, &s, &h->hash_rounds, nin_ids, nin_first, &n_owned_names));
        nin_first.release();
        KG_ALLOC(ctx, nmin, n_owned_names);
        KG_ALLOC(ctx, nhit, n_owned_names);
        KG_ALLOC(ctx, nlen, n_owned_names);
        KG_CUDA(ctx, cudaMemsetAsync(nmin.p, 0xff, (size_t)(n_owned_names ? n_owned_names : 1) * sizeof(unsigned long long), ctx->stream));
        KG_CUDA(ctx, cudaMemsetAsync(nhit.p, 0, (size_t)(n_owned_names ? n_owned_names : 1) * sizeof(uint32_t), ctx->stream));
        if (nin.n)
            KG_LAUNCH(ctx, name_merge_kernel, grid_for(nin.n, kThreads, ctx->sm_count), kThreads, 0, nin.msg, nin.n, nin_ids.p, nmin.p, nhit.p, nlen.p);
        // ---- 4. the names with a hit -> the homes of their first occurrences
        KG_TRY(outbox(n_owned_names));
        DevBuf<uint32_t> d_n(ctx, 1);
        if (!d_n) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
        KG_TRY((device_scan<uint32_t>(ctx, n_owned_names, UsedIn{nhit.p}, HitNameOut{nmin.p, nlen.p, d_cut.p, F, world, rank, out_msg.p, out_dest.p}, d_n.p)));
        return read_back(ctx, d_n.p, &n_hit_names, 1);
    }();
    Inbox hin;
    KG_TRY(send_msgs(c, rc, out_msg.p, out_dest.p, n_hit_names, nullptr, nullptr, &hin, kStage));
    // home: sort the keys it received, count them per (class, input)
    const int G = 2 * F;
    DevBuf<uint64_t> hkeys, htmp;
    DevBuf<unsigned long long> gcnt;
    uint64_t *hsorted = nullptr;
    std::vector<unsigned long long> mine((size_t)2 + G, 0ull), all;
    rc = [&]() -> int {
        KG_ALLOC(ctx, hkeys, hin.n);
        KG_ALLOC(ctx, htmp, hin.n);
        KG_ALLOC(ctx, gcnt, G ? G : 1);
        KG_CUDA(ctx, cudaMemsetAsync(gcnt.p, 0, (size_t)(G ? G : 1) * sizeof(unsigned long long), ctx->stream));
        if (hin.n) KG_LAUNCH(ctx, msg_keys_kernel, grid_for(hin.n, kThreads, ctx->sm_count), kThreads, 0, hin.msg, hin.n, F, hkeys.p, gcnt.p);
        uint64_t max_size = 0;
        for (int f = 0; f < F; ++f) max_size = sizes[f] > max_size ? sizes[f] : max_size;
        RadixPass passes[8];
        const int np = plan_radix_passes(0, bits_for(max_size), kKeyFileShift, 64, passes);
        KG_TRY(radix_sort_u64(ctx, hkeys.p, htmp.p, hin.n, passes, np, &hsorted));
        if (G) KG_TRY(read_back(ctx, gcnt.p, &mine[2], G));
        return KOMBGPU_OK;
    }();
    mine[1] = n_owned_names;
    KG_TRY(gather_words(c, rc, mine, all, kStage));
    const size_t k = 2 + (size_t)G;
    std::vector<unsigned long long> delta(G ? G : 1, 0);
    unsigned long long n_unitigs = 0, max_owned = 1;
    for (int g = 0; g < G; ++g) {
        unsigned long long before_me = 0, local_before = 0;
        for (int q = 0; q < world; ++q) {
            if (q < rank) before_me += all[q * k + 2 + g];
        }
        for (int g2 = 0; g2 < g; ++g2) local_before += mine[2 + g2];
        delta[g] = n_unitigs + before_me - local_before;
        for (int q = 0; q < world; ++q) n_unitigs += all[q * k + 2 + g];
    }
    for (int q = 0; q < world; ++q) max_owned = all[q * k + 1] > max_owned ? all[q * k + 1] : max_owned;
    if (n_unitigs >= 0xfffffffeull) return ctx_fail(ctx, KOMBGPU_EINVAL, "%llu unitigs exceed the 2^32 - 2 limit", n_unitigs);
    h->n_unitigs = (uint32_t)n_unitigs;
    const uint32_t step = owner_step(h->n_unitigs, world);
    uint32_t *vid_reply = nullptr, *sym_len = nullptr;
    uint64_t *sym_key = nullptr;
    PeerPtrs<uint32_t> pvid{}, plen{};
    PeerPtrs<uint64_t> pkey{};
    KG_TRY(sym_alloc(c, (size_t)max_owned, &vid_reply, &pvid));
    KG_TRY(sym_alloc(c, (size_t)step, &sym_key, &pkey));
    KG_TRY(sym_alloc(c, (size_t)step, &sym_len, &plen));
    rc = [&]() -> int {
        DevBuf<unsigned long long> d_delta;
        KG_ALLOC(ctx, d_delta, delta.size());
        KG_CUDA(ctx, cudaMemcpyAsync(d_delta.p, delta.data(), delta.size() * sizeof(unsigned long long), cudaMemcpyHostToDevice, ctx->stream));
        KG_TRY(outbox(hin.n));
        if (hin.n)
            KG_LAUNCH(ctx, vid_kernel, grid_for(hin.n, kThreads, ctx->sm_count), kThreads, 0, hin.msg, hin.n, hsorted, d_delta.p, F, step, pvid, pkey,
                      plen, Slices{d_base.p, d_cut_lo.p, F}, out_msg.p, out_dest.p, out_off.p);
        return KOMBGPU_OK;
    }();
    KG_TRY(barrier(c, rc, kStage));
    hkeys.release();
    htmp.release();
    // owner -> sender: the vid of every name it sent
    uint32_t *name_vid = nullptr;
    PeerPtrs<uint32_t> pname_vid{};
    KG_TRY(sym_alloc(c, (size_t)max_nd, &name_vid, &pname_vid));
    rc = [&]() -> int {
        if (nin.n)
            KG_LAUNCH(ctx, name_reply_kernel, grid_for(nin.n, kThreads, ctx->sm_count), kThreads, 0, nin.msg, nin.n, nin_ids.p, vid_reply, pname_vid);
        return KOMBGPU_OK;
    }();
    KG_TRY(barrier(c, rc, kStage));
    // home -> owner of the vid: the bytes of the name (a line is never split between slices, so the home holds them)
    Inbox bin;
    KG_TRY(send_msgs(c, KOMBGPU_OK, out_msg.p, out_dest.p, hin.n, text.p, out_off.p, &bin, kStage));
    DevBuf<unsigned char> name_bytes;
    DevBuf<uint64_t> name_off;
    rc = [&]() -> int {
        KG_ALLOC(ctx, name_bytes, bin.n_bytes);
        KG_ALLOC(ctx, name_off, bin.n);
        if (bin.n_bytes) KG_CUDA(ctx, cudaMemcpyAsync(name_bytes.p, bin.bytes, bin.n_bytes, cudaMemcpyDeviceToDevice, ctx->stream));
        if (bin.n) KG_LAUNCH(ctx, name_off_kernel, grid_for(bin.n, kThreads, ctx->sm_count), kThreads, 0, bin.msg, bin.n, name_off.p);
        return KOMBGPU_OK;
    }();
    h->ms_intern = tm.lap();

    // ---- 5. (read id << 32 | vid) of every hit -> the owner of the read
    DevBuf<uint64_t> hit_keys;
    if (rc == KOMBGPU_OK) rc = [&]() -> int {
        KG_ALLOC(ctx, hit_keys, n_hits);
        if (n_hits)
            KG_LAUNCH(ctx, hit_keys_kernel, grid_for(n_hits, kThreads, ctx->sm_count), kThreads, 0, key_ids.p, read_id, name_ids.p + n_sq, name_vid,
                      n_hits, hit_keys.p);
        return KOMBGPU_OK;
    }();
    uint64_t *recv = nullptr, n_recv = 0;
    KG_TRY(route_keys(c, hit_keys.p, rc == KOMBGPU_OK ? n_hits : 0, stride, false, &recv, &n_recv, rc));
    hit_keys.release();
    DevBuf<uint32_t> read_key, unitig, name_len;
    DevBuf<uint64_t> name_key;
    const uint64_t lo64 = (uint64_t)rank * step, hi64 = lo64 + step;
    h->v_lo = (uint32_t)(lo64 < n_unitigs ? lo64 : n_unitigs);
    h->n_local = (uint32_t)((hi64 < n_unitigs ? hi64 : n_unitigs) - h->v_lo);
    rc = [&]() -> int {
        KG_ALLOC(ctx, read_key, n_recv);
        KG_ALLOC(ctx, unitig, n_recv);
        KG_ALLOC(ctx, name_key, h->n_local);
        KG_ALLOC(ctx, name_len, h->n_local);
        if (n_recv) KG_LAUNCH(ctx, split_hits_kernel, grid_for(n_recv, kThreads, ctx->sm_count), kThreads, 0, recv, n_recv, read_key.p, unitig.p);
        if (h->n_local) {
            KG_CUDA(ctx, cudaMemcpyAsync(name_key.p, sym_key, h->n_local * sizeof(uint64_t), cudaMemcpyDeviceToDevice, ctx->stream));
            KG_CUDA(ctx, cudaMemcpyAsync(name_len.p, sym_len, h->n_local * sizeof(uint32_t), cudaMemcpyDeviceToDevice, ctx->stream));
        }
        return KOMBGPU_OK;
    }();
    {
        std::vector<unsigned long long> m2 = {0ull, n_recv}, a2;   // also the barrier after which the heap is reused
        KG_TRY(gather_words(c, rc, m2, a2, kStage));
        h->n_hits_global = 0;
        for (int q = 0; q < world; ++q) h->n_hits_global += a2[q * 2 + 1];
    }
    h->ms_route = tm.lap();
    h->n_hits_local = n_recv;
    h->read_key = read_key.take();
    h->unitig = unitig.take();
    h->name_key = name_key.take();
    h->name_len = name_len.take();
    h->name_bytes = name_bytes.take();
    h->name_off = name_off.take();
    return KOMBGPU_OK;
}

void dist_hits_release(kombgpu_dist_hits *h) {
    if (!h || !h->ctx) return;
    void *ptrs[] = {h->read_key, h->unitig, h->name_key, h->name_len, h->name_bytes, h->name_off};
    for (void *p : ptrs)
        if (p) ws_free(h->ctx, p);
    h->read_key = nullptr; h->unitig = nullptr; h->name_key = nullptr; h->name_len = nullptr; h->name_bytes = nullptr; h->name_off = nullptr;
}

}  // namespace

int dist_hits_name_text(const kombgpu_dist_hits *h, DistNames *out) {
    if (!h) return KOMBGPU_EINVAL;
    *out = DistNames{h->comm, h->n_unitigs, h->v_lo, h->n_local, h->name_bytes, h->name_off, h->name_len};
    return KOMBGPU_OK;
}
}  // namespace kg

using namespace kg;

extern "C" {

int kombgpu_dist_sam_parse(kombgpu_comm *c, const char *const *texts, const uint64_t *sizes, int n_files, kombgpu_dist_hits **out) {
    if (!c) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = c->ctx;
    // a bad argument is the caller's on every rank (every rank passes the same inputs): no rank waits for another
    if (!out || n_files < 0 || n_files > 64 || (n_files && (!texts || !sizes))) return ctx_fail(ctx, KOMBGPU_EINVAL, "bad argument");
    for (int f = 0; f < n_files; ++f)
        if (sizes[f] && !texts[f]) return ctx_fail(ctx, KOMBGPU_EINVAL, "null text with a non-zero size");
    *out = nullptr;
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    kombgpu_dist_hits *h = new (std::nothrow) kombgpu_dist_hits();
    if (!h) return ctx_fail(ctx, KOMBGPU_ENOMEM, "host allocation");
    h->comm = c;
    h->ctx = ctx;
    const int rc = dist_sam_parse(c, texts, sizes, n_files, h);
    if (rc != KOMBGPU_OK) {
        cudaStreamSynchronize(ctx->stream);
        dist_hits_release(h);
        delete h;
        return rc;
    }
    *out = h;
    return KOMBGPU_OK;
}

void kombgpu_dist_hits_destroy(kombgpu_dist_hits *h) {
    if (!h) return;
    dist_hits_release(h);
    delete h;
}

int kombgpu_dist_hits_counts(const kombgpu_dist_hits *h, uint64_t *n_hits_local, uint64_t *n_hits_global, uint32_t *n_reads_global,
                             uint32_t *n_unitigs, uint64_t *n_lines_global) {
    if (!h) return KOMBGPU_EINVAL;
    if (n_hits_local) *n_hits_local = h->n_hits_local;
    if (n_hits_global) *n_hits_global = h->n_hits_global;
    if (n_reads_global) *n_reads_global = h->n_reads_global;
    if (n_unitigs) *n_unitigs = h->n_unitigs;
    if (n_lines_global) *n_lines_global = h->n_lines_global;
    return KOMBGPU_OK;
}

int kombgpu_dist_hits_names(const kombgpu_dist_hits *h, uint32_t *file, uint64_t *offset, uint32_t *len) {
    if (!h) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = h->ctx;
    if (!offset || !len) return ctx_fail(ctx, KOMBGPU_EINVAL, "null argument");
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t n = h->n_local;
    if (n) {
        KG_CUDA(ctx, cudaMemcpyAsync(offset, h->name_key, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
        KG_CUDA(ctx, cudaMemcpyAsync(len, h->name_len, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
        KG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    for (size_t i = 0; i < n; ++i) {
        if (file) file[i] = (uint32_t)(offset[i] >> kKeyFileShift);
        offset[i] &= kKeyOffMask;
    }
    return KOMBGPU_OK;
}

int kombgpu_dist_hits_download(const kombgpu_dist_hits *h, uint32_t *read_key, uint32_t *unitig) {
    if (!h) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = h->ctx;
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    if (h->n_hits_local) {
        if (read_key) KG_CUDA(ctx, cudaMemcpyAsync(read_key, h->read_key, h->n_hits_local * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
        if (unitig) KG_CUDA(ctx, cudaMemcpyAsync(unitig, h->unitig, h->n_hits_local * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
        KG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return KOMBGPU_OK;
}

int kombgpu_dist_hits_device_arrays(const kombgpu_dist_hits *h, const uint32_t **read_key, const uint32_t **unitig) {
    if (!h) return KOMBGPU_EINVAL;
    if (read_key) *read_key = h->read_key;
    if (unitig) *unitig = h->unitig;
    return KOMBGPU_OK;
}

int kombgpu_dist_hits_timing(const kombgpu_dist_hits *h, float *ms_upload, float *ms_parse, float *ms_intern, float *ms_route, int *hash_rounds) {
    if (!h) return KOMBGPU_EINVAL;
    if (ms_upload) *ms_upload = h->ms_upload;
    if (ms_parse) *ms_parse = h->ms_parse;
    if (ms_intern) *ms_intern = h->ms_intern;
    if (ms_route) *ms_route = h->ms_route;
    if (hash_rounds) *hash_rounds = h->hash_rounds;
    return KOMBGPU_OK;
}

int kombgpu_dist_build_graph_hits(const kombgpu_dist_hits *h, kombgpu_dist_graph **out) {
    if (!h) return KOMBGPU_EINVAL;
    return kombgpu_dist_build_hits_dev(h->comm, h->read_key, h->unitig, h->n_hits_local, h->n_unitigs, out);
}

}  // extern "C"
