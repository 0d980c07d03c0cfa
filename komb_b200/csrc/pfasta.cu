// pfasta.cu — the unitig FASTA over the ranks of a communicator (kombgpu_dist_fasta_*, kombgpu_dist_anomalous; DESIGN.md
// §4 "Unitig FASTA").  Same records, names, join, fence and extraction as fasta.cu, whose kernels (fasta.cuh) do the
// work inside a rank; nothing of the file's size or of the vertex count passes through the host or one GPU:
//   load      rank q uploads and indexes only bytes [cut_q, cut_{q+1}) of the file, cut_q = the first record start at
//             or after floor(size q / world) (pmsg.cuh: a record is never split, a slice may be empty).  The ranks
//             exchange their record counts, so record ids are global.  Every record's name (bytes, global record id)
//             goes to its OWNER, the rank a fixed-seed hash of the bytes picks, which interns what it received by the
//             bytes (sam.cuh) and finds the repeated names.  The ranks agree on the first error in the single-GPU order
//   join      the name of every vertex of the rank's unitigs goes to the owner of its bytes; the owner interns its
//             record names and the received vertex names together and stores the record id, or kMissing, into the
//             sender's reply slot (symmetric heap)
//   extract   the rank of each selected vertex stores a 1 into the `sel` byte of its record on the rank that holds the
//             record (symmetric heap); after one barrier every rank copies its own selected records (copy_selected)
//   fence     a radix select over the ranks finds the four order statistics the quartiles need: 8-bit digits of the
//             scores' order-preserving images, every rank histograms its own keys under the agreed prefixes, the ranks
//             sum the histograms through peer memory.  No score crosses a link.  fasta.cuh's fence_from then gives
//             q1, q3 and the fence bit for bit as on one GPU
// Kernels only store to and load from peer buffers; none waits for a peer, so ranks that share one device work too.
#include <algorithm>
#include <new>
#include <string>
#include <vector>

#include "dgraph.cuh"
#include "fasta.cuh"
#include "pmsg.cuh"
#include "sam.cuh"

struct kombgpu_dist_fasta {
    kombgpu_comm *comm = nullptr;
    kombgpu_ctx *ctx = nullptr;
    uint64_t size = 0, byte_lo = 0, byte_hi = 0;   // the file; this rank's slice is bytes [byte_lo, byte_hi)
    uint32_t n_rec = 0, n_rec_global = 0;          // the slice's records are global records [rec_lo[rank], rec_lo[rank + 1])
    std::vector<uint32_t> rec_lo;                  // [world + 1]
    bool unterminated = false;             // the slice holds the file's last record, which does not end in '\n'
    unsigned char *text = nullptr;         // the slice, zero padded to a multiple of 16 bytes plus 16 more
    uint64_t *rec_start = nullptr;         // [n_rec + 1] offset of every record's '>' in the slice; rec_start[n_rec] = its size
    // the record names this rank owns: bytes [own_off[i], own_off[i] + own_len[i]) of own_bytes name global record own_rec[i]
    unsigned char *own_bytes = nullptr;
    uint64_t *own_off = nullptr;
    uint32_t *own_len = nullptr, *own_rec = nullptr;
    uint64_t n_own = 0, n_own_bytes = 0;
    // last join: this rank's vertices [v_lo, v_lo + n_local)
    bool joined = false;
    uint32_t v_lo = 0, n_local = 0;
    uint32_t *vrec = nullptr;              // [n_local] global record of every vertex, kMissing when the FASTA has none
    std::vector<uint32_t> missing;         // local vertices without a record, ascending
    std::vector<uint64_t> missing_off;     // their names: bytes [missing_off[i], missing_off[i + 1]) of missing_names
    std::string missing_names;
    // last extraction: this rank's slice of the output
    bool extracted = false;
    char *out = nullptr;
    uint64_t out_bytes = 0;
    float ms_upload = 0.f, ms_index = 0.f, ms_join = 0.f, ms_extract = 0.f;
    uint64_t launches = 0;
};

namespace kg {
namespace {

constexpr uint64_t kOwnerSeed = 0x2545f4914f6cdd1dull;   // picks a name's owner: the same on every rank, never changed
constexpr const char *kStage = "the unitig FASTA call";    // named in the error of a rank whose peer failed
constexpr int kNameWords = 26;                            // 208 bytes: enough of a name for printable()'s 200 and its "..."

// record r of the slice -> message to the owner of its name: key = the name's global byte offset, idx = global record
// id.  flag[0] = smallest local record with an empty name
__global__ void __launch_bounds__(kThreads) record_msgs_kernel(const unsigned char *__restrict__ text, const uint64_t *__restrict__ start,
                                                               uint32_t n_rec, uint64_t byte_lo, uint32_t rec_lo, int world, int rank,
                                                               Msg *__restrict__ msg, uint32_t *__restrict__ dest, uint64_t *__restrict__ src_off,
                                                               uint32_t *__restrict__ flag) {
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n_rec; r += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t lo = start[r] + 1;
        const uint32_t len = record_name_len(text, lo, start[r + 1]);
        if (len == 0) atomicMin(flag, (uint32_t)r);
        dest[r] = (uint32_t)(hash_span(text + lo, len, kOwnerSeed) % (uint64_t)world);
        msg[r] = Msg{byte_lo + lo, 0ull, len, rec_lo + (uint32_t)r, (uint32_t)rank, 0u};
        src_off[r] = lo;
    }
}

// vertex v's name -> message to its owner (the bytes stay where they are: send_msgs reads them at nm.off[v])
__global__ void __launch_bounds__(kThreads) vertex_msgs_kernel(NameSpans nm, uint32_t n, int world, int rank, Msg *__restrict__ msg,
                                                               uint32_t *__restrict__ dest) {
    for (uint64_t v = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; v < n; v += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t len = nm.length((uint32_t)v);
        dest[v] = (uint32_t)(hash_span(nm.text + nm.off[v], len, kOwnerSeed) % (uint64_t)world);
        msg[v] = Msg{0ull, 0ull, len, (uint32_t)v, (uint32_t)rank, 0u};
    }
}

// the received strings as spans of a byte buffer in which they start at byte `base`; rec (optional) = their idx
__global__ void __launch_bounds__(kThreads) inbox_spans_kernel(const Msg *__restrict__ msg, uint64_t n, uint64_t base, uint64_t *__restrict__ off,
                                                               uint32_t *__restrict__ len, uint32_t *__restrict__ rec) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        off[i] = base + msg[i].off;
        len[i] = msg[i].len;
        if (rec) rec[i] = msg[i].idx;
    }
}

// owner: the smallest record of every distinct name, then the smallest record that repeats an earlier one
__global__ void __launch_bounds__(kThreads) name_min_kernel(const uint32_t *__restrict__ ids, const uint32_t *__restrict__ rec, uint64_t n,
                                                            uint32_t *__restrict__ min_rec) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) atomicMin(&min_rec[ids[i]], rec[i]);
}
__global__ void __launch_bounds__(kThreads) name_dup_kernel(const uint32_t *__restrict__ ids, const uint32_t *__restrict__ rec, uint64_t n,
                                                            const uint32_t *__restrict__ min_rec, uint32_t *__restrict__ dup) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
        if (rec[i] != min_rec[ids[i]]) atomicMin(dup, rec[i]);
}
// ... and where that record's name starts in the file: the key of its message
__global__ void __launch_bounds__(kThreads) find_rec_kernel(const Msg *__restrict__ msg, uint64_t n, uint32_t r, unsigned long long *__restrict__ at) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
        if (msg[i].idx == r) { at[0] = msg[i].key; at[1] = msg[i].len; }
}

// owner, join: the record of every distinct name (items [0, n_rec) are its record names), then the reply to every
// vertex name it received (items n_rec ...): the record, or kMissing
__global__ void __launch_bounds__(kThreads) rec_of_kernel(const uint32_t *__restrict__ ids, const uint32_t *__restrict__ rec, uint64_t n_rec,
                                                          uint32_t *__restrict__ rec_of) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_rec; i += (uint64_t)gridDim.x * blockDim.x) rec_of[ids[i]] = rec[i];
}
__global__ void __launch_bounds__(kThreads) join_reply_kernel(const Msg *__restrict__ msg, uint64_t n, const uint32_t *__restrict__ ids,
                                                              const uint32_t *__restrict__ rec_of, PeerPtrs<uint32_t> reply) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
        reply.p[msg[i].rank][msg[i].idx] = rec_of[ids[i]];
}

struct RecLo {   // the first global record of every rank's slice, [world + 1]
    uint32_t lo[kMaxRanks + 1];
    int world;
};

// the rank of each selected vertex marks its record in the sel array of the rank that holds the record
__global__ void __launch_bounds__(kThreads) dist_mark_kernel(const uint8_t *__restrict__ mask, uint32_t n, const uint32_t *__restrict__ vrec, RecLo rl,
                                                             PeerPtrs<uint8_t> sel, uint32_t *__restrict__ missing_selected) {
    for (uint64_t v = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; v < n; v += (uint64_t)gridDim.x * blockDim.x) {
        if (!mask[v]) continue;
        const uint32_t r = vrec[v];
        if (r == kMissing) { atomicMin(missing_selected, (uint32_t)v); continue; }
        int q = 0;   // the last rank whose slice starts at or before r (empty slices start where the next one does)
        for (int k = 1; k < rl.world; ++k)
            if (rl.lo[k] <= r) q = k;
        sel.p[q][r - rl.lo[q]] = 1;
    }
}

// ---- the fence: radix select of four order statistics over the ranks
constexpr int kDigitBits = 8, kBins = 1 << kDigitBits, kStats = 4;

struct Prefixes {   // the digits decided so far of each wanted order statistic
    uint64_t p[kStats];
};

// hist[t][b] += keys whose decided digits are those of statistic t and whose digit at `shift` is b
__global__ void __launch_bounds__(kThreads) radix_hist_kernel(const uint64_t *__restrict__ key, uint32_t n, Prefixes pre, int shift,
                                                              uint32_t *__restrict__ hist) {
    __shared__ uint32_t h[kStats * kBins];
    for (int i = threadIdx.x; i < kStats * kBins; i += blockDim.x) h[i] = 0;
    __syncthreads();
    const int hi = shift + kDigitBits;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t k = key[i];
        const uint32_t b = (uint32_t)(k >> shift) & (kBins - 1);
#pragma unroll
        for (int t = 0; t < kStats; ++t)
            if (hi >= 64 || (k >> hi) == (pre.p[t] >> hi)) atomicAdd(&h[t * kBins + b], 1u);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < kStats * kBins; i += blockDim.x)
        if (h[i]) atomicAdd(&hist[i], h[i]);
}
// the histograms of all ranks, summed (loads from peer memory)
__global__ void __launch_bounds__(kThreads) hist_sum_kernel(PeerPtrs<uint32_t> hist, size_t at, int world, uint32_t *__restrict__ sum) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < kStats * kBins; i += gridDim.x * blockDim.x) {
        uint32_t s = 0;
        for (int q = 0; q < world; ++q) s += hist.p[q][at + i];
        sum[i] = s;
    }
}
__global__ void fence_positions_kernel(uint32_t n, uint32_t *__restrict__ pos) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    double t[2];
    fence_positions(n, pos, t);
}
__global__ void fence_stats_kernel(Prefixes stat, uint32_t n, double whisker, double *__restrict__ out) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    fence_from(stat.p, n, whisker, out);
}

// ---- load + index
void dist_fasta_release_join(kombgpu_dist_fasta *fa) {
    if (fa->vrec) ws_free(fa->ctx, fa->vrec);
    if (fa->out) ws_free(fa->ctx, fa->out);
    fa->vrec = nullptr;
    fa->out = nullptr;
    fa->joined = fa->extracted = false;
    fa->v_lo = fa->n_local = 0;
    fa->out_bytes = 0;
    fa->missing.clear();
    fa->missing_off.clear();
    fa->missing_names.clear();
}

void dist_fasta_release(kombgpu_dist_fasta *fa) {
    if (!fa || !fa->ctx) return;
    dist_fasta_release_join(fa);
    void *ptrs[] = {fa->text, fa->rec_start, fa->own_bytes, fa->own_off, fa->own_len, fa->own_rec};
    for (void *p : ptrs)
        if (p) ws_free(fa->ctx, p);
    fa->text = nullptr; fa->rec_start = nullptr; fa->own_bytes = nullptr; fa->own_off = nullptr; fa->own_len = nullptr; fa->own_rec = nullptr;
}

int dist_fasta_load(kombgpu_comm *c, const char *src, uint64_t size, kombgpu_dist_fasta *fa) {
    kombgpu_ctx *ctx = c->ctx;
    const int world = c->world, rank = c->rank;
    SymRewind heap{c, sym_mark(c)};
    EvTimer tm(ctx);
    const uint64_t launches0 = ctx->launches;
    std::vector<uint64_t> cut;
    slice_cuts(&src, &size, 1, world, '>', cut);
    const uint64_t lo = cut[rank], len = cut[rank + 1] - lo, padded = (len + 15) & ~15ull, chunks = padded / 16;
    fa->size = size;
    fa->byte_lo = lo;
    fa->byte_hi = lo + len;

    // ---- 1. upload the slice, count its records, check the bytes before the first one
    DevBuf<unsigned char> text;
    DevBuf<unsigned long long> d_cnt;   // [starts, first start, first non-blank byte before it]
    unsigned long long h_cnt[3] = {0ull, ~0ull, ~0ull};
    const uint4 *t4 = nullptr;
    int rc = [&]() -> int {
        KG_ALLOC(ctx, text, padded + 16);
        t4 = reinterpret_cast<const uint4 *>(text.p);
        if (len) KG_CUDA(ctx, cudaMemcpyAsync(text.p, src + lo, len, cudaMemcpyHostToDevice, ctx->stream));
        KG_CUDA(ctx, cudaMemsetAsync(text.p + len, 0, padded + 16 - len, ctx->stream));
        fa->ms_upload = tm.lap();
        KG_ALLOC(ctx, d_cnt, 3);
        KG_CUDA(ctx, cudaMemsetAsync(d_cnt.p, 0, sizeof(unsigned long long), ctx->stream));
        KG_CUDA(ctx, cudaMemsetAsync(d_cnt.p + 1, 0xff, 2 * sizeof(unsigned long long), ctx->stream));
        // offset 0 of a slice counts as a line start: it is the file's, or a record start that follows a '\n'
        if (chunks) KG_LAUNCH(ctx, fasta_starts_count_kernel, grid_for(chunks, kThreads * 4, ctx->sm_count), kThreads, 0, t4, chunks, d_cnt.p);
        KG_TRY(read_back(ctx, d_cnt.p, h_cnt, 2));
        const uint64_t first = h_cnt[0] ? h_cnt[1] : len;
        if (first) {   // only rank 0's slice can hold bytes before the first record
            KG_LAUNCH(ctx, fasta_prefix_check_kernel, grid_for(first, kThreads, ctx->sm_count), kThreads, 0, text.p, first, d_cnt.p + 2);
            KG_TRY(read_back(ctx, d_cnt.p + 2, &h_cnt[2], 1));
        }
        return KOMBGPU_OK;
    }();
    {
        std::vector<unsigned long long> mine = {0ull, h_cnt[0], h_cnt[2] == ~0ull ? ~0ull : lo + h_cnt[2]}, all;
        KG_TRY(gather_words(c, rc, mine, all, kStage));
        unsigned long long total = 0, bad = ~0ull;
        fa->rec_lo.assign((size_t)world + 1, 0);
        for (int q = 0; q < world; ++q) {
            fa->rec_lo[q] = (uint32_t)std::min<unsigned long long>(total, 0xffffffffull);
            total += all[(size_t)q * 3 + 1];
            bad = std::min(bad, all[(size_t)q * 3 + 2]);
        }
        if (total >= 0xffffffffull) return ctx_fail(ctx, KOMBGPU_EINVAL, "%llu FASTA records exceed the 2^32 - 1 limit", total);
        if (bad != ~0ull)
            return ctx_fail(ctx, KOMBGPU_EINVAL, "malformed FASTA: byte %llu (0x%02x) comes before the first record ('>' at a line start)", bad,
                            (unsigned)(unsigned char)src[bad]);
        fa->rec_lo[world] = (uint32_t)total;
        fa->n_rec_global = (uint32_t)total;
    }
    const uint32_t n_rec = (uint32_t)h_cnt[0], rec_lo = fa->rec_lo[rank];
    fa->n_rec = n_rec;
    fa->unterminated = n_rec && fa->byte_hi == size && src[size - 1] != '\n';

    // ---- 2. record starts; every record's name -> its owner
    DevBuf<uint64_t> rec_start, out_off;
    DevBuf<Msg> out_msg;
    DevBuf<uint32_t> out_dest, d_flag;
    uint32_t empty_local = kMissing;
    rc = [&]() -> int {
        KG_ALLOC(ctx, rec_start, (size_t)n_rec + 1);
        KG_CUDA(ctx, cudaMemcpyAsync(rec_start.p + n_rec, &len, sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream));
        if (n_rec) KG_TRY((device_scan<uint64_t>(ctx, chunks, StartsIn{t4}, StartsOut{t4, rec_start.p}, (uint64_t *)nullptr)));
        KG_ALLOC(ctx, out_msg, n_rec);
        KG_ALLOC(ctx, out_dest, n_rec);
        KG_ALLOC(ctx, out_off, n_rec);
        KG_ALLOC(ctx, d_flag, 1);
        KG_CUDA(ctx, cudaMemsetAsync(d_flag.p, 0xff, sizeof(uint32_t), ctx->stream));
        if (n_rec)
            KG_LAUNCH(ctx, record_msgs_kernel, grid_for(n_rec, kThreads, ctx->sm_count), kThreads, 0, text.p, rec_start.p, n_rec, lo, rec_lo, world, rank,
                      out_msg.p, out_dest.p, out_off.p, d_flag.p);
        return read_back(ctx, d_flag.p, &empty_local, 1);
    }();
    Inbox in;
    KG_TRY(send_msgs(c, rc, out_msg.p, out_dest.p, rc == KOMBGPU_OK ? n_rec : 0, text.p, out_off.p, &in, kStage));

    // ---- 3. owner: intern the names it received, find the repeated ones; keep them for the joins
    DevBuf<unsigned char> own_bytes;
    DevBuf<uint64_t> own_off;
    DevBuf<uint32_t> own_len, own_rec;
    unsigned long long empty_at = ~0ull, dup_at[2] = {~0ull, 0ull};
    uint32_t dup = kMissing;
    rc = [&]() -> int {
        KG_ALLOC(ctx, own_bytes, in.n_bytes);
        KG_ALLOC(ctx, own_off, in.n);
        KG_ALLOC(ctx, own_len, in.n);
        KG_ALLOC(ctx, own_rec, in.n);
        if (in.n_bytes) KG_CUDA(ctx, cudaMemcpyAsync(own_bytes.p, in.bytes, in.n_bytes, cudaMemcpyDeviceToDevice, ctx->stream));
        DevBuf<uint64_t> hash;
        KG_ALLOC(ctx, hash, in.n);
        const Items it{own_off.p, hash.p, own_len.p};
        uint64_t seed = 0x9e3779b97f4a7c15ull;
        int rounds = 0;
        DevBuf<uint32_t> ids, first, min_rec, d_dup(ctx, 1);
        DevBuf<unsigned long long> d_at(ctx, 2);
        if (!d_dup || !d_at) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
        KG_CUDA(ctx, cudaMemsetAsync(d_dup.p, 0xff, sizeof(uint32_t), ctx->stream));
        if (in.n) {
            const uint32_t grid = grid_for(in.n, kThreads, ctx->sm_count);
            KG_LAUNCH(ctx, inbox_spans_kernel, grid, kThreads, 0, in.msg, in.n, 0ull, own_off.p, own_len.p, own_rec.p);
            KG_LAUNCH(ctx, rehash_kernel, grid, kThreads, 0, own_bytes.p, it, in.n, seed);
        }
        uint32_t n_distinct = 0;
        KG_TRY(intern_items(ctx, own_bytes.p, it, in.n, &seed, &rounds, ids, first, &n_distinct));
        KG_ALLOC(ctx, min_rec, n_distinct);
        if (in.n) {
            const uint32_t grid = grid_for(in.n, kThreads, ctx->sm_count);
            KG_CUDA(ctx, cudaMemsetAsync(min_rec.p, 0xff, (size_t)n_distinct * sizeof(uint32_t), ctx->stream));
            KG_LAUNCH(ctx, name_min_kernel, grid, kThreads, 0, ids.p, own_rec.p, in.n, min_rec.p);
            KG_LAUNCH(ctx, name_dup_kernel, grid, kThreads, 0, ids.p, own_rec.p, in.n, min_rec.p, d_dup.p);
            KG_TRY(read_back(ctx, d_dup.p, &dup, 1));
            if (dup != kMissing) {
                KG_LAUNCH(ctx, find_rec_kernel, grid, kThreads, 0, in.msg, in.n, dup, d_at.p);
                KG_TRY(read_back(ctx, d_at.p, dup_at, 2));
            }
        }
        if (empty_local != kMissing) {
            uint64_t at = 0;
            KG_TRY(read_back(ctx, rec_start.p + empty_local, &at, 1));
            empty_at = lo + at;
        }
        return KOMBGPU_OK;
    }();
    {
        // the first error in the single-GPU order: the smallest record with an empty name, then the smallest record
        // that repeats the name of an earlier one
        std::vector<unsigned long long> mine = {0ull, empty_local == kMissing ? ~0ull : (unsigned long long)rec_lo + empty_local, empty_at,
                                                dup == kMissing ? ~0ull : (unsigned long long)dup, dup_at[0], dup_at[1]},
                                        all;
        KG_TRY(gather_words(c, rc, mine, all, kStage));
        int e = -1, d = -1;
        for (int q = 0; q < world; ++q) {
            if (all[(size_t)q * 6 + 1] != ~0ull && (e < 0 || all[(size_t)q * 6 + 1] < all[(size_t)e * 6 + 1])) e = q;
            if (all[(size_t)q * 6 + 3] != ~0ull && (d < 0 || all[(size_t)q * 6 + 3] < all[(size_t)d * 6 + 3])) d = q;
        }
        if (e >= 0)
            return ctx_fail(ctx, KOMBGPU_EINVAL, "malformed FASTA: record %u (byte %llu) has an empty name", (uint32_t)all[(size_t)e * 6 + 1],
                            all[(size_t)e * 6 + 2]);
        if (d >= 0) {
            const std::string name(src + all[(size_t)d * 6 + 4], (size_t)all[(size_t)d * 6 + 5]);
            return ctx_fail(ctx, KOMBGPU_EINVAL, "malformed FASTA: record %u repeats the name '%s' of an earlier record", (uint32_t)all[(size_t)d * 6 + 3],
                            printable(name).c_str());
        }
    }
    fa->ms_index = tm.lap();
    fa->launches += ctx->launches - launches0;
    fa->text = text.take();
    fa->rec_start = rec_start.take();
    fa->own_bytes = own_bytes.take();
    fa->own_off = own_off.take();
    fa->own_len = own_len.take();
    fa->own_rec = own_rec.take();
    fa->n_own = in.n;
    fa->n_own_bytes = in.n_bytes;
    return KOMBGPU_OK;
}

// ---- join.  rc: this rank's arguments were already refused with that code (it still takes part, so no rank waits)
int dist_fasta_join(kombgpu_dist_fasta *fa, int rc, NameSpans nm, uint32_t n, uint32_t *n_missing) {
    kombgpu_comm *c = fa->comm;
    kombgpu_ctx *ctx = fa->ctx;
    const int world = c->world, rank = c->rank;
    SymRewind heap{c, sym_mark(c)};
    EvTimer tm(ctx);
    const uint64_t launches0 = ctx->launches;
    dist_fasta_release_join(fa);
    if (rc != KOMBGPU_OK) n = 0;
    uint32_t v_lo = 0, max_n = 1;
    {
        std::vector<unsigned long long> mine = {0ull, n}, all;
        KG_TRY(gather_words(c, rc, mine, all, kStage));
        unsigned long long sum = 0;
        for (int q = 0; q < world; ++q) {
            if (q == rank) v_lo = (uint32_t)std::min<unsigned long long>(sum, 0xffffffffull);
            sum += all[(size_t)q * 2 + 1];
            max_n = std::max<uint32_t>(max_n, (uint32_t)all[(size_t)q * 2 + 1]);
        }
        if (sum > 0xffffffffull) return ctx_fail(ctx, KOMBGPU_EINVAL, "%llu vertices over the ranks exceed 32-bit ids", sum);
    }
    // ---- every vertex name -> its owner
    DevBuf<Msg> msg;
    DevBuf<uint32_t> dest;
    rc = [&]() -> int {
        KG_ALLOC(ctx, msg, n);
        KG_ALLOC(ctx, dest, n);
        if (n) KG_LAUNCH(ctx, vertex_msgs_kernel, grid_for(n, kThreads, ctx->sm_count), kThreads, 0, nm, n, world, rank, msg.p, dest.p);
        return KOMBGPU_OK;
    }();
    Inbox in;
    KG_TRY(send_msgs(c, rc, msg.p, dest.p, rc == KOMBGPU_OK ? n : 0, nm.text, nm.off, &in, kStage));
    // ---- owner: its record names and the received vertex names interned together; the record of each goes back
    uint32_t *reply = nullptr;
    PeerPtrs<uint32_t> preply{};
    KG_TRY(sym_alloc(c, (size_t)max_n, &reply, &preply));
    rc = [&]() -> int {
        const uint64_t n_items = fa->n_own + in.n;
        DevBuf<unsigned char> bytes;
        ItemBufs it;
        KG_ALLOC(ctx, bytes, fa->n_own_bytes + in.n_bytes);
        KG_TRY(it.alloc(ctx, n_items));
        if (fa->n_own_bytes) KG_CUDA(ctx, cudaMemcpyAsync(bytes.p, fa->own_bytes, fa->n_own_bytes, cudaMemcpyDeviceToDevice, ctx->stream));
        if (in.n_bytes) KG_CUDA(ctx, cudaMemcpyAsync(bytes.p + fa->n_own_bytes, in.bytes, in.n_bytes, cudaMemcpyDeviceToDevice, ctx->stream));
        if (fa->n_own) {
            KG_CUDA(ctx, cudaMemcpyAsync(it.off.p, fa->own_off, fa->n_own * sizeof(uint64_t), cudaMemcpyDeviceToDevice, ctx->stream));
            KG_CUDA(ctx, cudaMemcpyAsync(it.len.p, fa->own_len, fa->n_own * sizeof(uint32_t), cudaMemcpyDeviceToDevice, ctx->stream));
        }
        if (in.n)
            KG_LAUNCH(ctx, inbox_spans_kernel, grid_for(in.n, kThreads, ctx->sm_count), kThreads, 0, in.msg, in.n, fa->n_own_bytes, it.off.p + fa->n_own,
                      it.len.p + fa->n_own, (uint32_t *)nullptr);
        uint64_t seed = 0x9e3779b97f4a7c15ull;
        int rounds = 0;
        if (n_items) KG_LAUNCH(ctx, rehash_kernel, grid_for(n_items, kThreads, ctx->sm_count), kThreads, 0, bytes.p, it.view(), n_items, seed);
        DevBuf<uint32_t> ids, first, rec_of;
        uint32_t n_distinct = 0;
        KG_TRY(intern_items(ctx, bytes.p, it.view(), n_items, &seed, &rounds, ids, first, &n_distinct));
        KG_ALLOC(ctx, rec_of, n_distinct);
        if (n_distinct) KG_CUDA(ctx, cudaMemsetAsync(rec_of.p, 0xff, (size_t)n_distinct * sizeof(uint32_t), ctx->stream));
        if (fa->n_own)
            KG_LAUNCH(ctx, rec_of_kernel, grid_for(fa->n_own, kThreads, ctx->sm_count), kThreads, 0, ids.p, fa->own_rec, fa->n_own, rec_of.p);
        if (in.n)
            KG_LAUNCH(ctx, join_reply_kernel, grid_for(in.n, kThreads, ctx->sm_count), kThreads, 0, in.msg, in.n, ids.p + fa->n_own, rec_of.p, preply);
        return KOMBGPU_OK;
    }();
    KG_TRY(barrier(c, rc, kStage));   // every reply has landed
    DevBuf<uint32_t> vrec, d_miss(ctx, 1);
    uint32_t miss = 0;
    rc = [&]() -> int {
        KG_ALLOC(ctx, vrec, n);
        if (!d_miss) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
        KG_CUDA(ctx, cudaMemsetAsync(d_miss.p, 0, sizeof(uint32_t), ctx->stream));
        if (n) {
            KG_CUDA(ctx, cudaMemcpyAsync(vrec.p, reply, (size_t)n * sizeof(uint32_t), cudaMemcpyDeviceToDevice, ctx->stream));
            KG_TRY((device_scan<uint32_t>(ctx, n, MissingFlagIn{vrec.p}, NoOp{}, d_miss.p)));
        }
        KG_TRY(read_back(ctx, d_miss.p, &miss, 1));
        if (miss) KG_TRY(missing_to_host(ctx, nm, vrec.p, n, miss, fa->missing, fa->missing_off, fa->missing_names));
        return KOMBGPU_OK;
    }();
    unsigned long long total = 0;
    {
        std::vector<unsigned long long> mine = {0ull, miss}, all;   // also the barrier after which the heap is reused
        KG_TRY(gather_words(c, rc, mine, all, kStage));
        for (int q = 0; q < world; ++q) total += all[(size_t)q * 2 + 1];
    }
    fa->ms_join = tm.lap();
    fa->launches += ctx->launches - launches0;
    fa->vrec = vrec.take();
    fa->v_lo = v_lo;
    fa->n_local = n;
    fa->joined = true;
    *n_missing = (uint32_t)total;
    return KOMBGPU_OK;
}

int dist_fasta_extract(kombgpu_dist_fasta *fa, int rc, const uint8_t *mask, uint64_t *bytes) {
    kombgpu_comm *c = fa->comm;
    kombgpu_ctx *ctx = fa->ctx;
    const int world = c->world, rank = c->rank;
    SymRewind heap{c, sym_mark(c)};
    EvTimer tm(ctx);
    const uint64_t launches0 = ctx->launches;
    const uint32_t n = rc == KOMBGPU_OK ? fa->n_local : 0, n_rec = fa->n_rec;
    if (fa->out) ws_free(ctx, fa->out);
    fa->out = nullptr;
    fa->out_bytes = 0;
    fa->extracted = false;
    uint32_t max_rec = 1;
    RecLo rl{};
    rl.world = world;
    for (int q = 0; q <= world; ++q) rl.lo[q] = fa->rec_lo[q];
    for (int q = 0; q < world; ++q) max_rec = std::max(max_rec, rl.lo[q + 1] - rl.lo[q]);
    uint8_t *sel = nullptr;
    PeerPtrs<uint8_t> psel{};
    KG_TRY(sym_alloc(c, (size_t)max_rec, &sel, &psel));
    DevBuf<uint8_t> d_mask;
    DevBuf<uint32_t> d_err;
    if (rc == KOMBGPU_OK) rc = [&]() -> int {
        KG_ALLOC(ctx, d_mask, n);
        KG_ALLOC(ctx, d_err, 1);
        if (n) KG_CUDA(ctx, cudaMemcpyAsync(d_mask.p, mask, n, cudaMemcpyHostToDevice, ctx->stream));
        KG_CUDA(ctx, cudaMemsetAsync(sel, 0, max_rec, ctx->stream));
        KG_CUDA(ctx, cudaMemsetAsync(d_err.p, 0xff, sizeof(uint32_t), ctx->stream));
        return KOMBGPU_OK;
    }();
    KG_TRY(barrier(c, rc, kStage));   // every sel is clear before any rank marks
    uint32_t bad = kMissing;
    rc = [&]() -> int {
        if (n) KG_LAUNCH(ctx, dist_mark_kernel, grid_for(n, kThreads, ctx->sm_count), kThreads, 0, d_mask.p, n, fa->vrec, rl, psel, d_err.p);
        return read_back(ctx, d_err.p, &bad, 1);
    }();
    int who = -1;
    unsigned long long bad_vid = ~0ull;
    {
        std::vector<unsigned long long> mine = {0ull, bad == kMissing ? ~0ull : (unsigned long long)fa->v_lo + bad}, all;   // every mark has landed
        KG_TRY(gather_words(c, rc, mine, all, kStage));
        for (int q = 0; q < world; ++q)
            if (all[(size_t)q * 2 + 1] < bad_vid) { bad_vid = all[(size_t)q * 2 + 1]; who = q; }
    }
    if (who >= 0) {
        // the smallest selected vertex without a record, and (from the rank that owns it) the start of its name
        std::vector<unsigned long long> mine(2 + kNameWords, 0ull), all;
        if (who == rank) {
            const size_t i = (size_t)(std::lower_bound(fa->missing.begin(), fa->missing.end(), bad) - fa->missing.begin());
            const std::string name = i < fa->missing.size() ? fa->missing_names.substr(fa->missing_off[i], fa->missing_off[i + 1] - fa->missing_off[i]) : "";
            const size_t k = std::min(name.size(), (size_t)kNameWords * 8);
            mine[1] = k;
            memcpy(&mine[2], name.data(), k);
        }
        KG_TRY(gather_words(c, KOMBGPU_OK, mine, all, kStage));
        const unsigned long long *w = &all[(size_t)who * (2 + kNameWords)];
        const std::string name(reinterpret_cast<const char *>(w + 2), (size_t)w[1]);
        return ctx_fail(ctx, KOMBGPU_EINVAL, "selected vertex %u (unitig '%s') has no record in the FASTA", (uint32_t)bad_vid, printable(name).c_str());
    }
    char *out = nullptr;
    uint64_t total = 0;
    rc = copy_selected(ctx, fa->text, fa->rec_start, sel, n_rec, fa->unterminated ? n_rec - 1 : kMissing, &out, &total);
    KG_TRY(barrier(c, rc, kStage));   // no rank reuses the heap while another still reads its sel
    fa->ms_extract = tm.lap();
    fa->launches += ctx->launches - launches0;
    fa->out = out;
    fa->out_bytes = total;
    fa->extracted = true;
    *bytes = total;
    return KOMBGPU_OK;
}

// ---- the IQR fence over the scores of all ranks
int dist_anomalous(kombgpu_dist_graph *g, double whisker, double *q1, double *q3, double *fence, uint32_t *n_selected, uint8_t *member) {
    kombgpu_comm *c = g->comm;
    kombgpu_ctx *ctx = g->ctx;
    const int world = c->world;
    const uint32_t n_local = g->n_local;
    SymRewind heap{c, sym_mark(c)};
    DevBuf<uint64_t> key;
    DevBuf<uint32_t> flags;
    uint32_t nan_seen = 0;
    const uint32_t grid = grid_for(n_local, kThreads, ctx->sm_count);
    int rc = [&]() -> int {
        KG_ALLOC(ctx, key, n_local);
        KG_ALLOC(ctx, flags, 2);
        KG_CUDA(ctx, cudaMemsetAsync(flags.p, 0, 2 * sizeof(uint32_t), ctx->stream));
        if (n_local) KG_LAUNCH(ctx, score_keys_kernel, grid, kThreads, 0, g->score, n_local, key.p, flags.p);
        return read_back(ctx, flags.p, &nan_seen, 1);
    }();
    unsigned long long n = 0;
    {
        std::vector<unsigned long long> mine = {0ull, nan_seen, n_local}, all;
        KG_TRY(gather_words(c, rc, mine, all, kStage));
        bool nan_any = false;
        for (int q = 0; q < world; ++q) {
            nan_any |= all[(size_t)q * 3 + 1] != 0;
            n += all[(size_t)q * 3 + 2];
        }
        if (nan_any) return ctx_fail(ctx, KOMBGPU_EINVAL, "a score is NaN: the quartiles are undefined");
    }
    double q[3] = {0.0, 0.0, 0.0};
    uint32_t cnt = 0;
    if (n) {
        // the positions of the four order statistics, from the same arithmetic as fence_kernel
        uint32_t pos[kStats] = {0, 0, 0, 0};
        DevBuf<uint32_t> d_pos, d_sum;
        rc = [&]() -> int {
            KG_ALLOC(ctx, d_pos, kStats);
            KG_ALLOC(ctx, d_sum, kStats * kBins);
            KG_LAUNCH(ctx, fence_positions_kernel, 1, 32, 0, (uint32_t)n, d_pos.p);
            return read_back(ctx, d_pos.p, pos, kStats);
        }();
        uint32_t *hist = nullptr;   // two histogram buffers, used by turns: one barrier per digit
        PeerPtrs<uint32_t> phist{};
        KG_TRY(sym_alloc(c, (size_t)2 * kStats * kBins, &hist, &phist));
        Prefixes pre{};
        uint64_t rank_in[kStats];
        for (int t = 0; t < kStats; ++t) rank_in[t] = pos[t];
        std::vector<uint32_t> sum(kStats * kBins);
        for (int d = 0; d < 64 / kDigitBits; ++d) {
            const int shift = 64 - kDigitBits * (d + 1);
            const size_t at = (size_t)(d & 1) * kStats * kBins;
            if (rc == KOMBGPU_OK) rc = [&]() -> int {
                KG_CUDA(ctx, cudaMemsetAsync(hist + at, 0, kStats * kBins * sizeof(uint32_t), ctx->stream));
                if (n_local) KG_LAUNCH(ctx, radix_hist_kernel, grid, kThreads, 0, key.p, n_local, pre, shift, hist + at);
                return KOMBGPU_OK;
            }();
            KG_TRY(barrier(c, rc, kStage));
            rc = [&]() -> int {
                KG_LAUNCH(ctx, hist_sum_kernel, 4, kThreads, 0, phist, at, world, d_sum.p);
                return read_back(ctx, d_sum.p, sum.data(), sum.size());
            }();
            for (int t = 0; t < kStats && rc == KOMBGPU_OK; ++t) {
                uint64_t below = 0;
                int b = 0;
                while (b < kBins - 1 && below + sum[(size_t)t * kBins + b] <= rank_in[t]) below += sum[(size_t)t * kBins + b++];
                rank_in[t] -= below;
                pre.p[t] |= (uint64_t)b << shift;
            }
        }
        DevBuf<double> dq;
        DevBuf<uint8_t> dm;
        rc = [&]() -> int {
            KG_TRY(rc);
            KG_ALLOC(ctx, dq, 3);
            KG_ALLOC(ctx, dm, n_local);
            KG_CUDA(ctx, cudaMemsetAsync(flags.p + 1, 0, sizeof(uint32_t), ctx->stream));
            KG_LAUNCH(ctx, fence_stats_kernel, 1, 32, 0, pre, (uint32_t)n, whisker, dq.p);
            if (n_local) KG_LAUNCH(ctx, member_kernel, grid, kThreads, 0, g->score, n_local, dq.p, dm.p, flags.p + 1);
            KG_TRY(read_back(ctx, dq.p, q, 3));
            KG_TRY(read_back(ctx, flags.p + 1, &cnt, 1));
            if (member && n_local) {
                KG_CUDA(ctx, cudaMemcpyAsync(member, dm.p, n_local, cudaMemcpyDeviceToHost, ctx->stream));
                KG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
            }
            return KOMBGPU_OK;
        }();
        std::vector<unsigned long long> mine = {0ull, cnt}, all;   // also the barrier after which the heap is reused
        KG_TRY(gather_words(c, rc, mine, all, kStage));
        cnt = 0;
        for (int k = 0; k < world; ++k) cnt += (uint32_t)all[(size_t)k * 2 + 1];
    }
    if (q1) *q1 = q[0];
    if (q3) *q3 = q[1];
    if (fence) *fence = q[2];
    if (n_selected) *n_selected = cnt;
    return KOMBGPU_OK;
}

}  // namespace
}  // namespace kg

using namespace kg;

extern "C" {

int kombgpu_dist_fasta_load(kombgpu_comm *c, const char *text, uint64_t size, kombgpu_dist_fasta **out) {
    if (!c) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = c->ctx;
    // a bad argument is the caller's on every rank (every rank passes the same bytes): no rank waits for another
    if (!out || (size && !text)) return ctx_fail(ctx, KOMBGPU_EINVAL, "null argument");
    *out = nullptr;
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    kombgpu_dist_fasta *fa = new (std::nothrow) kombgpu_dist_fasta();
    if (!fa) return ctx_fail(ctx, KOMBGPU_ENOMEM, "host allocation");
    fa->comm = c;
    fa->ctx = ctx;
    const int rc = dist_fasta_load(c, text, size, fa);
    if (rc != KOMBGPU_OK) {
        cudaStreamSynchronize(ctx->stream);
        dist_fasta_release(fa);
        delete fa;
        return rc;
    }
    *out = fa;
    return KOMBGPU_OK;
}

void kombgpu_dist_fasta_destroy(kombgpu_dist_fasta *fa) {
    if (!fa) return;
    if (fa->ctx) cudaSetDevice(fa->ctx->device);
    dist_fasta_release(fa);
    delete fa;
}

int kombgpu_dist_fasta_counts(const kombgpu_dist_fasta *fa, uint32_t *n_records_local, uint32_t *n_records_global, uint32_t *rec_lo,
                              uint64_t *byte_lo, uint64_t *byte_hi) {
    if (!fa) return KOMBGPU_EINVAL;
    if (n_records_local) *n_records_local = fa->n_rec;
    if (n_records_global) *n_records_global = fa->n_rec_global;
    if (rec_lo) *rec_lo = fa->rec_lo[fa->comm->rank];
    if (byte_lo) *byte_lo = fa->byte_lo;
    if (byte_hi) *byte_hi = fa->byte_hi;
    return KOMBGPU_OK;
}

int kombgpu_dist_fasta_join_hits(kombgpu_dist_fasta *fa, const kombgpu_dist_hits *names, uint32_t *n_missing) {
    if (!fa) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = fa->ctx;
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    DistNames dn{};
    int rc = KOMBGPU_OK;
    uint32_t scratch = 0;
    if (!n_missing || !names || dist_hits_name_text(names, &dn) != KOMBGPU_OK) rc = ctx_fail(ctx, KOMBGPU_EINVAL, "null argument");
    else if (dn.comm != fa->comm) rc = ctx_fail(ctx, KOMBGPU_EINVAL, "the names belong to another communicator");
    const int jrc = dist_fasta_join(fa, rc, NameSpans{dn.bytes, dn.off, dn.len}, rc == KOMBGPU_OK ? dn.n_local : 0, n_missing ? n_missing : &scratch);
    return rc != KOMBGPU_OK ? rc : jrc;
}

int kombgpu_dist_fasta_join_names(kombgpu_dist_fasta *fa, const char *bytes, const uint64_t *offsets, uint32_t n_local, uint32_t *n_missing) {
    if (!fa) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = fa->ctx;
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc = KOMBGPU_OK;
    uint32_t scratch = 0;
    if (!n_missing || !offsets || (offsets[n_local] && !bytes)) rc = ctx_fail(ctx, KOMBGPU_EINVAL, "null argument");
    for (uint32_t v = 0; rc == KOMBGPU_OK && v < n_local; ++v)
        if (offsets[v + 1] < offsets[v] || offsets[v + 1] - offsets[v] > 0xffffffffull)
            rc = ctx_fail(ctx, KOMBGPU_EINVAL, "name offsets must not decrease (entry %u)", v + 1);
    DevBuf<unsigned char> d_bytes;
    DevBuf<uint64_t> d_off;
    if (rc == KOMBGPU_OK) rc = [&]() -> int {
        const uint64_t total = offsets[n_local];
        KG_ALLOC(ctx, d_bytes, total);
        KG_ALLOC(ctx, d_off, (size_t)n_local + 1);
        if (total) KG_CUDA(ctx, cudaMemcpyAsync(d_bytes.p, bytes, total, cudaMemcpyHostToDevice, ctx->stream));
        KG_CUDA(ctx, cudaMemcpyAsync(d_off.p, offsets, ((size_t)n_local + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream));
        return KOMBGPU_OK;
    }();
    const int jrc = dist_fasta_join(fa, rc, NameSpans{d_bytes.p, d_off.p, nullptr}, rc == KOMBGPU_OK ? n_local : 0, n_missing ? n_missing : &scratch);
    return rc != KOMBGPU_OK ? rc : jrc;
}

int kombgpu_dist_fasta_extract(kombgpu_dist_fasta *fa, const uint8_t *mask, uint32_t n_local, uint64_t *bytes) {
    if (!fa) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = fa->ctx;
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc = KOMBGPU_OK;
    uint64_t scratch = 0;
    if (!fa->joined) rc = ctx_fail(ctx, KOMBGPU_ESTATE, "kombgpu_dist_fasta_extract needs a join first");
    else if (!bytes || (n_local && !mask)) rc = ctx_fail(ctx, KOMBGPU_EINVAL, "null argument");
    else if (n_local != fa->n_local) rc = ctx_fail(ctx, KOMBGPU_EINVAL, "the mask has %u entries, the last join %u vertices on this rank", n_local, fa->n_local);
    const int erc = dist_fasta_extract(fa, rc, mask, bytes ? bytes : &scratch);
    return rc != KOMBGPU_OK ? rc : erc;
}

int kombgpu_dist_fasta_extract_fetch(kombgpu_dist_fasta *fa, char *dst) {
    if (!fa) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = fa->ctx;
    if (!fa->extracted) return ctx_fail(ctx, KOMBGPU_ESTATE, "kombgpu_dist_fasta_extract has not run");
    if (!fa->out_bytes) return KOMBGPU_OK;
    if (!dst) return ctx_fail(ctx, KOMBGPU_EINVAL, "null destination");
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    KG_CUDA(ctx, cudaMemcpyAsync(dst, fa->out, fa->out_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    KG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return KOMBGPU_OK;
}

int kombgpu_dist_fasta_timing(const kombgpu_dist_fasta *fa, float *ms_upload, float *ms_index, float *ms_join, float *ms_extract,
                              uint64_t *kernel_launches) {
    if (!fa) return KOMBGPU_EINVAL;
    if (ms_upload) *ms_upload = fa->ms_upload;
    if (ms_index) *ms_index = fa->ms_index;
    if (ms_join) *ms_join = fa->ms_join;
    if (ms_extract) *ms_extract = fa->ms_extract;
    if (kernel_launches) *kernel_launches = fa->launches;
    return KOMBGPU_OK;
}

int kombgpu_dist_anomalous(kombgpu_dist_graph *g, double whisker, double *q1, double *q3, double *fence, uint32_t *n_selected, uint8_t *member) {
    if (!g) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = g->ctx;
    if (!g->has_score) return ctx_fail(ctx, KOMBGPU_ESTATE, "kombgpu_dist_anomalous needs the CORE-A scores (kombgpu_dist_corea) first");
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    return dist_anomalous(g, whisker, q1, q3, fence, n_selected, member);
}

}  // extern "C"
