// fasta.cu — the unitig FASTA on the device: index its records, join them to the graph's vertices by name, pick the
// anomalous unitigs (IQR fence on CORE-A) and copy the selected records out (include/kombgpu.h, unitig FASTA).
//
// Kernels (all HBM-bound byte / integer work):
//   index     fasta_starts_count_kernel: 16 bytes per thread (one uint4), SIMD byte compares, counts the record starts
//             ('>' at offset 0 or after '\n') and finds the first; one scan then writes the starts; bytes before the
//             first record are checked only when there are any
//   names     fasta_name_insert_kernel: one thread per record walks its name (up to the first whitespace byte),
//             hashes it and inserts the hash into an open-addressing table (CAS; the slot keeps the smallest record
//             index); fasta_name_verify_kernel compares every record's name BYTES with the first record of its slot:
//             different bytes are a 64-bit collision (the pass repeats with another seed), equal bytes a duplicate name
//   join      fasta_probe_kernel: one thread per vertex name (a span of the SAM text the graph came from, or of an
//             uploaded host table) probes the table and compares bytes; a slot holds one distinct name, so an equal
//             hash with different bytes means "no record", never a wrong record
//   select    the scores' order-preserving u64 images through radix_sort_u64, the quartiles and the fence in one
//             thread (numpy's "linear" percentile, operation by operation, no contraction), then one pass for the mask
//   extract   the mask is scattered through vertex -> record; one scan places the selected records in the output (as
//             format.cu places rows), one more lists them as pieces of at most kPiece bytes; one warp per piece copies
//             with 16-byte stores at aligned destinations (source words realigned with funnel shifts)
#include <algorithm>
#include <new>
#include <string>
#include <vector>

#include "graph.cuh"
#include "primitives.cuh"
#include "strings.cuh"

struct kombgpu_hits;
namespace kg { int hits_name_spans(const kombgpu_hits *h, kombgpu_ctx **ctx, const unsigned char **text, const uint64_t **off, const uint32_t **len,
                                   uint32_t *n_unitigs); }

struct kombgpu_fasta {
    kombgpu_ctx *ctx = nullptr;
    unsigned char *text = nullptr;          // the file, zero padded to a multiple of 16 bytes plus 16 more
    uint64_t size = 0;
    uint32_t n_rec = 0;
    bool unterminated = false;              // the last record does not end in '\n'
    uint64_t *rec_start = nullptr;          // [n_rec + 1] offset of every record's '>'; rec_start[n_rec] = size
    uint32_t *name_len = nullptr;           // [n_rec] the name is bytes [rec_start + 1, rec_start + 1 + name_len)
    unsigned long long *tab_key = nullptr;  // [cap] name hash per slot (0 = empty)
    uint32_t *tab_rec = nullptr;            // [cap] the record whose name has that hash
    uint32_t cap_mask = 0;
    int shift = 0;
    uint64_t seed = 0;
    // last join
    bool joined = false;
    uint32_t n_vertices = 0;
    uint32_t *vrec = nullptr;               // [n_vertices] record of every vertex, kMissing when the FASTA has none
    std::vector<uint32_t> missing;          // vertices without a record, ascending
    std::vector<uint64_t> missing_off;      // their names: bytes [missing_off[i], missing_off[i + 1]) of missing_names
    std::string missing_names;
    // last extraction
    bool extracted = false;
    char *out = nullptr;
    uint64_t out_bytes = 0;
    float ms_upload = 0.f, ms_index = 0.f, ms_join = 0.f, ms_extract = 0.f;
    uint64_t launches = 0;
};

namespace kg {
namespace {

constexpr int kThreads = 256;
constexpr uint32_t kMissing = 0xffffffffu;
constexpr uint64_t kPiece = 16384;   // bytes one warp copies at a time: long records are split into pieces of this size

inline uint32_t grid_for(uint64_t n, int per_block, int sms) {
    const uint64_t g = (n + per_block - 1) / per_block;
    const uint64_t cap = (uint64_t)sms * 16u;
    return (uint32_t)(g < 1 ? 1 : (g > cap ? cap : g));
}

// bit j set when byte j of the 16 equals the byte repeated in pat
__device__ __forceinline__ uint32_t byte_mask16(uint4 w, uint32_t pat) {
    const uint32_t ws[4] = {w.x, w.y, w.z, w.w};
    uint32_t m = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint32_t e = __vcmpeq4(ws[k], pat);
        m |= (((e >> 7) & 1u) | ((e >> 14) & 2u) | ((e >> 21) & 4u) | ((e >> 28) & 8u)) << (4 * k);
    }
    return m;
}
// record starts inside chunk c: '>' at offset 0 of the file or right after a '\n'
__device__ __forceinline__ uint32_t starts_in(const uint4 *t, uint4 w, uint64_t c) {
    const uint32_t prev_nl = c == 0 ? 1u : (reinterpret_cast<const unsigned char *>(t)[c * 16 - 1] == '\n' ? 1u : 0u);
    return byte_mask16(w, 0x3e3e3e3eu) & ((byte_mask16(w, 0x0a0a0a0au) << 1) | prev_nl) & 0xffffu;
}

__device__ __forceinline__ bool is_space(unsigned char b) { return b == ' ' || b == '\t' || b == '\r' || b == '\n' || b == '\v' || b == '\f'; }

// cnt[0] = number of record starts, cnt[1] = offset of the first one (init ~0)
__global__ void __launch_bounds__(kThreads) fasta_starts_count_kernel(const uint4 *__restrict__ text, uint64_t n_chunks,
                                                                      unsigned long long *__restrict__ cnt) {
    uint32_t c_here = 0;
    unsigned long long first = ~0ull;
    for (uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; c < n_chunks; c += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t m = starts_in(text, ld_stream_u4(text + c), c);
        if (m && first == ~0ull) first = c * 16 + (__ffs(m) - 1);
        c_here += __popc(m);
    }
    c_here = warp_reduce_add(c_here);
    first = warp_reduce_min(first);
    if (lane_id() == 0) {
        if (c_here) atomicAdd(&cnt[0], (unsigned long long)c_here);
        if (first != ~0ull) atomicMin(&cnt[1], first);
    }
}

struct StartsIn {
    const uint4 *text;
    __device__ uint64_t operator()(uint64_t c) const { return __popc(starts_in(text, text[c], c)); }
};
struct StartsOut {
    const uint4 *text;
    uint64_t *start;
    __device__ void operator()(uint64_t c, uint64_t prefix, uint64_t cnt) const {
        if (!cnt) return;
        uint32_t m = starts_in(text, text[c], c);
        uint64_t k = prefix;
        while (m) {
            const int j = __ffs(m) - 1;
            m &= m - 1;
            start[k++] = c * 16 + (uint64_t)j;
        }
    }
};

// *bad = smallest offset in [0, end) of a byte that is not whitespace
__global__ void __launch_bounds__(kThreads) fasta_prefix_check_kernel(const unsigned char *__restrict__ text, uint64_t end,
                                                                      unsigned long long *__restrict__ bad) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < end; i += (uint64_t)gridDim.x * blockDim.x)
        if (!is_space(text[i])) atomicMin(bad, (unsigned long long)i);
}

struct NameTable {
    unsigned long long *key;
    uint32_t *rec;
    uint32_t cap_mask;
    int shift;
    __device__ __forceinline__ uint32_t home(unsigned long long h) const { return (uint32_t)((h * 0x9e3779b97f4a7c15ull) >> shift) & cap_mask; }
};

// flags[0] = smallest record with an empty name, flags[1] = collision seen, flags[2] = smallest record whose name an
// earlier record already has
__global__ void __launch_bounds__(kThreads) fasta_name_insert_kernel(const unsigned char *__restrict__ text, const uint64_t *__restrict__ start,
                                                                     uint32_t n_rec, uint64_t seed, NameTable tab, uint32_t *__restrict__ name_len,
                                                                     uint32_t *__restrict__ slot_of, uint32_t *__restrict__ flags) {
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n_rec; r += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t lo = start[r] + 1, end = start[r + 1];
        uint64_t p = lo;
        while (p < end && !is_space(text[p])) ++p;
        const uint32_t len = (uint32_t)(p - lo);
        name_len[r] = len;
        if (len == 0) atomicMin(&flags[0], (uint32_t)r);
        unsigned long long h = hash_span(text + lo, len, seed);
        if (h == 0) h = 1;   // 0 marks an empty slot
        uint32_t slot = tab.home(h);
        while (true) {
            const unsigned long long old = atomicCAS(&tab.key[slot], 0ull, h);
            if (old == 0ull || old == h) break;
            slot = (slot + 1u) & tab.cap_mask;
        }
        atomicMin(&tab.rec[slot], (uint32_t)r);
        slot_of[r] = slot;
    }
}

__device__ __forceinline__ bool same_bytes(const unsigned char *a, const unsigned char *b, uint32_t len) {
    for (uint32_t k = 0; k < len; ++k)
        if (a[k] != b[k]) return false;
    return true;
}

__global__ void __launch_bounds__(kThreads) fasta_name_verify_kernel(const unsigned char *__restrict__ text, const uint64_t *__restrict__ start,
                                                                     const uint32_t *__restrict__ name_len, uint32_t n_rec, const uint32_t *__restrict__ tab_rec,
                                                                     const uint32_t *__restrict__ slot_of, uint32_t *__restrict__ flags) {
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n_rec; r += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t f = tab_rec[slot_of[r]];
        if (f == (uint32_t)r) continue;
        const uint32_t len = name_len[r];
        if (len == name_len[f] && same_bytes(text + start[r] + 1, text + start[f] + 1, len)) atomicMin(&flags[2], (uint32_t)r);
        else atomicExch(&flags[1], 1u);
    }
}

// names of the vertices: bytes [off[v], off[v] + len[v]) of `text`, or [off[v], off[v + 1]) when len is null
struct NameSpans {
    const unsigned char *text;
    const uint64_t *off;
    const uint32_t *len;
    __device__ __forceinline__ uint32_t length(uint32_t v) const { return len ? len[v] : (uint32_t)(off[v + 1] - off[v]); }
};

__global__ void __launch_bounds__(kThreads) fasta_probe_kernel(NameSpans nm, uint32_t n, const unsigned char *__restrict__ text,
                                                               const uint64_t *__restrict__ start, const uint32_t *__restrict__ name_len, NameTable tab,
                                                               uint64_t seed, uint32_t *__restrict__ vrec, uint32_t *__restrict__ n_missing) {
    uint32_t miss = 0;
    for (uint64_t v = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; v < n; v += (uint64_t)gridDim.x * blockDim.x) {
        const unsigned char *p = nm.text + nm.off[v];
        const uint32_t len = nm.length((uint32_t)v);
        unsigned long long h = hash_span(p, len, seed);
        if (h == 0) h = 1;
        uint32_t slot = tab.home(h), rec = kMissing;
        while (true) {
            const unsigned long long k = tab.key[slot];
            if (k == 0ull) break;
            if (k == h) {
                const uint32_t r = tab.rec[slot];
                if (name_len[r] == len && same_bytes(p, text + start[r] + 1, len)) rec = r;
                break;   // the slot holds the only record name with this hash
            }
            slot = (slot + 1u) & tab.cap_mask;
        }
        vrec[v] = rec;
        miss += rec == kMissing ? 1u : 0u;
    }
    miss = warp_reduce_add(miss);
    if (lane_id() == 0 && miss) atomicAdd(n_missing, miss);
}

// the names of the missing vertices, packed: one scan sizes them, one thread per name copies
struct MissingFlagIn {
    const uint32_t *vrec;
    __device__ uint32_t operator()(uint64_t v) const { return vrec[v] == kMissing ? 1u : 0u; }
};
struct MissingListOut {
    uint32_t *ids;
    __device__ void operator()(uint64_t v, uint32_t pos, uint32_t flag) const { if (flag) ids[pos] = (uint32_t)v; }
};
struct MissingLenIn {
    NameSpans nm;
    const uint32_t *ids;
    __device__ uint64_t operator()(uint64_t i) const { return nm.length(ids[i]); }
};
struct MissingNameOut {
    NameSpans nm;
    const uint32_t *ids;
    uint64_t *off;
    char *bytes;
    __device__ void operator()(uint64_t i, uint64_t at, uint64_t len) const {
        off[i] = at;
        const unsigned char *p = nm.text + nm.off[ids[i]];
        for (uint64_t k = 0; k < len; ++k) bytes[at + k] = (char)p[k];
    }
};

struct NoOp {
    __device__ void operator()(uint64_t, uint64_t, uint64_t) const {}
};

// ---- extraction
__global__ void __launch_bounds__(kThreads) fasta_mark_kernel(const uint8_t *__restrict__ mask, uint32_t n, const uint32_t *__restrict__ vrec,
                                                              uint8_t *__restrict__ sel, uint32_t *__restrict__ missing_selected) {
    for (uint64_t v = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; v < n; v += (uint64_t)gridDim.x * blockDim.x) {
        if (!mask[v]) continue;
        const uint32_t r = vrec[v];
        if (r == kMissing) atomicMin(missing_selected, (uint32_t)v);
        else sel[r] = 1;
    }
}

// bytes of record r in the output: the record, plus the '\n' appended to an unterminated last record
struct OutLenIn {
    const uint8_t *sel;
    const uint64_t *start;
    uint32_t nl_rec;   // the unterminated last record, or kMissing
    __device__ uint64_t operator()(uint64_t r) const {
        return sel[r] ? start[r + 1] - start[r] + (r == nl_rec ? 1ull : 0ull) : 0ull;
    }
};
struct OutOffOut {
    uint64_t *out_off;
    __device__ void operator()(uint64_t r, uint64_t at, uint64_t) const { out_off[r] = at; }
};
struct PiecesIn {
    const uint8_t *sel;
    const uint64_t *start;
    __device__ uint64_t operator()(uint64_t r) const { return sel[r] ? (start[r + 1] - start[r] + kPiece - 1) / kPiece : 0ull; }
};
struct PiecesOut {
    uint64_t *first_piece;
    uint32_t *piece_rec;
    __device__ void operator()(uint64_t r, uint64_t at, uint64_t cnt) const {
        first_piece[r] = at;
        for (uint64_t k = 0; k < cnt; ++k) piece_rec[at + k] = (uint32_t)r;
    }
};

// 16 bytes starting at byte s (0..15) of the 32 bytes a:b
__device__ __forceinline__ uint4 realign16(uint4 a, uint4 b, uint32_t s) {
    const uint32_t q = s >> 2, sh = 8u * (s & 3u);
    const uint32_t w0 = q == 0 ? a.x : q == 1 ? a.y : q == 2 ? a.z : a.w;
    const uint32_t w1 = q == 0 ? a.y : q == 1 ? a.z : q == 2 ? a.w : b.x;
    const uint32_t w2 = q == 0 ? a.z : q == 1 ? a.w : q == 2 ? b.x : b.y;
    const uint32_t w3 = q == 0 ? a.w : q == 1 ? b.x : q == 2 ? b.y : b.z;
    const uint32_t w4 = q == 0 ? b.x : q == 1 ? b.y : q == 2 ? b.z : b.w;
    return make_uint4(__funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh), __funnelshift_r(w2, w3, sh), __funnelshift_r(w3, w4, sh));
}

// one warp per piece; the text buffer holds 16 readable bytes past its last aligned word
__global__ void __launch_bounds__(kThreads) fasta_copy_kernel(const unsigned char *__restrict__ text, const uint64_t *__restrict__ start,
                                                              const uint64_t *__restrict__ out_off, const uint64_t *__restrict__ first_piece,
                                                              const uint32_t *__restrict__ piece_rec, uint64_t n_pieces, uint32_t nl_rec,
                                                              char *__restrict__ out) {
    const uint32_t lane = lane_id();
    const uint64_t warps = (uint64_t)gridDim.x * (blockDim.x / 32);
    for (uint64_t p = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) / 32; p < n_pieces; p += warps) {
        const uint32_t r = piece_rec[p];
        const uint64_t k = p - first_piece[r];
        const uint64_t rec_end = start[r + 1];
        const uint64_t src = start[r] + k * kPiece;
        const uint64_t len = min(kPiece, rec_end - src);
        const uint64_t dst = out_off[r] + k * kPiece;
        const uint64_t head = min(len, (16u - (dst & 15u)) & 15u);
        const uint64_t n_words = (len - head) / 16, tail = (len - head) % 16;
        if (lane < head) out[dst + lane] = (char)text[src + lane];
        const uint64_t s0 = src + head;
        const uint32_t s = (uint32_t)(s0 & 15u);
        const uint4 *t4 = reinterpret_cast<const uint4 *>(text) + (s0 >> 4);
        uint4 *o4 = reinterpret_cast<uint4 *>(out + dst + head);
        for (uint64_t w = lane; w < n_words; w += 32) {
            const uint4 a = __ldg(t4 + w);
            o4[w] = s ? realign16(a, __ldg(t4 + w + 1), s) : a;
        }
        const uint64_t t0 = head + n_words * 16;
        if (lane < tail) out[dst + t0 + lane] = (char)text[src + t0 + lane];
        if (r == nl_rec && src + len == rec_end && lane == 0) out[dst + len] = '\n';
    }
}

// ---- anomalous unitigs
// order-preserving image of a double: negative values bit-flipped, the others with the sign bit set
__global__ void __launch_bounds__(kThreads) score_keys_kernel(const double *__restrict__ score, uint32_t n, uint64_t *__restrict__ key,
                                                              uint32_t *__restrict__ nan_seen) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const double x = score[i];
        if (x != x) atomicExch(nan_seen, 1u);
        const uint64_t b = (uint64_t)__double_as_longlong(x);
        key[i] = (b >> 63) ? ~b : (b | (1ull << 63));
    }
}
__device__ __forceinline__ double key_value(uint64_t k) {
    return __longlong_as_double((long long)((k >> 63) ? (k & ~(1ull << 63)) : ~k));
}

// numpy.percentile(s, 100 p, method="linear") of the sorted scores, with numpy's operations in numpy's order (the
// _rn intrinsics keep the compiler from contracting a multiply and an add into one rounding)
__device__ double quartile(const uint64_t *sorted, uint32_t n, double p) {
    const double h = __dsub_rn(__dmul_rn((double)n, p), p);
    const double fi = floor(h);
    const uint32_t i = (uint32_t)fi, j = min(i + 1u, n - 1u);
    const double t = __dsub_rn(h, fi);
    const double si = key_value(sorted[i]), sj = key_value(sorted[j]);
    const double d = __dsub_rn(sj, si);
    return t < 0.5 ? __dadd_rn(si, __dmul_rn(d, t)) : __dsub_rn(sj, __dmul_rn(d, __dsub_rn(1.0, t)));
}
// out = {q1, q3, fence}
__global__ void fence_kernel(const uint64_t *__restrict__ sorted, uint32_t n, double whisker, double *__restrict__ out) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    const double q1 = quartile(sorted, n, 0.25), q3 = quartile(sorted, n, 0.75);
    out[0] = q1;
    out[1] = q3;
    out[2] = __dadd_rn(q3, __dmul_rn(whisker, __dsub_rn(q3, q1)));
}
__global__ void __launch_bounds__(kThreads) member_kernel(const double *__restrict__ score, uint32_t n, const double *__restrict__ fence,
                                                          uint8_t *__restrict__ member, uint32_t *__restrict__ count) {
    const double f = fence[2];
    uint32_t c = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const bool m = score[i] > f;
        member[i] = m ? 1 : 0;
        c += m ? 1u : 0u;
    }
    c = warp_reduce_add(c);
    if (lane_id() == 0 && c) atomicAdd(count, c);
}

int anomalous_dev(kombgpu_ctx *ctx, const double *score, uint32_t n, double whisker, double *q1, double *q3, double *fence,
                  uint32_t *n_selected, uint8_t *member) {
    double q[3] = {0.0, 0.0, 0.0};
    uint32_t cnt = 0;
    if (n) {
        DevBuf<uint64_t> ka, kb;
        DevBuf<uint32_t> flags(ctx, 2);
        DevBuf<double> dq(ctx, 3);
        DevBuf<uint8_t> dm;
        KG_ALLOC(ctx, ka, n);
        KG_ALLOC(ctx, kb, n);
        KG_ALLOC(ctx, dm, n);
        if (!flags || !dq) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
        KG_CUDA(ctx, cudaMemsetAsync(flags.p, 0, 2 * sizeof(uint32_t), ctx->stream));
        const uint32_t grid = grid_for(n, kThreads, ctx->sm_count);
        KG_LAUNCH(ctx, score_keys_kernel, grid, kThreads, 0, score, n, ka.p, flags.p);
        uint32_t nan_seen = 0;
        KG_TRY(read_back(ctx, flags.p, &nan_seen, 1));
        if (nan_seen) return ctx_fail(ctx, KOMBGPU_EINVAL, "a score is NaN: the quartiles are undefined");
        RadixPass passes[8];
        const int np = plan_radix_passes(0, 64, 0, 0, passes);
        uint64_t *sorted = nullptr;
        KG_TRY(radix_sort_u64(ctx, ka.p, kb.p, n, passes, np, &sorted));
        KG_LAUNCH(ctx, fence_kernel, 1, 32, 0, sorted, n, whisker, dq.p);
        KG_LAUNCH(ctx, member_kernel, grid, kThreads, 0, score, n, dq.p, dm.p, flags.p + 1);
        KG_TRY(read_back(ctx, dq.p, q, 3));
        KG_TRY(read_back(ctx, flags.p + 1, &cnt, 1));
        if (member) {
            KG_CUDA(ctx, cudaMemcpyAsync(member, dm.p, n, cudaMemcpyDeviceToHost, ctx->stream));
            KG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        }
    }
    if (q1) *q1 = q[0];
    if (q3) *q3 = q[1];
    if (fence) *fence = q[2];
    if (n_selected) *n_selected = cnt;
    return KOMBGPU_OK;
}

// ---- load + index
void fasta_release_join(kombgpu_fasta *fa) {
    if (fa->vrec) ws_free(fa->ctx, fa->vrec);
    if (fa->out) ws_free(fa->ctx, fa->out);
    fa->vrec = nullptr;
    fa->out = nullptr;
    fa->joined = fa->extracted = false;
    fa->n_vertices = 0;
    fa->out_bytes = 0;
    fa->missing.clear();
    fa->missing_off.clear();
    fa->missing_names.clear();
}

void fasta_release(kombgpu_fasta *fa) {
    if (!fa || !fa->ctx) return;
    fasta_release_join(fa);
    void *ptrs[] = {fa->text, fa->rec_start, fa->name_len, fa->tab_key, fa->tab_rec};
    for (void *p : ptrs)
        if (p) ws_free(fa->ctx, p);
    fa->text = nullptr; fa->rec_start = nullptr; fa->name_len = nullptr; fa->tab_key = nullptr; fa->tab_rec = nullptr;
}

std::string printable(const std::string &s) {
    std::string o;
    for (unsigned char c : s.substr(0, 200)) {
        if (c >= 0x20 && c < 0x7f) o += (char)c;
        else { char b[8]; snprintf(b, sizeof b, "\\x%02x", c); o += b; }
    }
    return s.size() > 200 ? o + "..." : o;
}

int fasta_load(kombgpu_ctx *ctx, const char *src, uint64_t size, kombgpu_fasta *fa) {
    cudaEvent_t e0 = ctx->ev_a, e1 = ctx->ev_b;
    const uint64_t launches0 = ctx->launches;
    const uint64_t padded = (size + 15) & ~15ull;
    fa->size = size;
    DevBuf<unsigned char> text;
    KG_ALLOC(ctx, text, padded + 16);
    KG_CUDA(ctx, cudaEventRecord(e0, ctx->stream));
    if (size) KG_CUDA(ctx, cudaMemcpyAsync(text.p, src, size, cudaMemcpyHostToDevice, ctx->stream));
    KG_CUDA(ctx, cudaMemsetAsync(text.p + size, 0, padded + 16 - size, ctx->stream));
    KG_CUDA(ctx, cudaEventRecord(e1, ctx->stream));
    KG_CUDA(ctx, cudaEventSynchronize(e1));
    cudaEventElapsedTime(&fa->ms_upload, e0, e1);
    KG_CUDA(ctx, cudaEventRecord(e0, ctx->stream));

    // ---- record starts
    const uint64_t chunks = padded / 16;
    const uint4 *t4 = reinterpret_cast<const uint4 *>(text.p);
    DevBuf<unsigned long long> d_cnt(ctx, 3);   // [starts, first start, first non-blank byte before it]
    if (!d_cnt) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
    KG_CUDA(ctx, cudaMemsetAsync(d_cnt.p, 0, sizeof(unsigned long long), ctx->stream));
    KG_CUDA(ctx, cudaMemsetAsync(d_cnt.p + 1, 0xff, 2 * sizeof(unsigned long long), ctx->stream));
    if (chunks) KG_LAUNCH(ctx, fasta_starts_count_kernel, grid_for(chunks, kThreads * 4, ctx->sm_count), kThreads, 0, t4, chunks, d_cnt.p);
    unsigned long long h_cnt[2] = {0, 0};
    KG_TRY(read_back(ctx, d_cnt.p, h_cnt, 2));
    const uint64_t first = h_cnt[0] ? h_cnt[1] : size;
    if (h_cnt[0] >= 0xffffffffull) return ctx_fail(ctx, KOMBGPU_EINVAL, "%llu FASTA records exceed the 2^32 - 1 limit", h_cnt[0]);
    if (first) {
        KG_LAUNCH(ctx, fasta_prefix_check_kernel, grid_for(first, kThreads, ctx->sm_count), kThreads, 0, text.p, first, d_cnt.p + 2);
        unsigned long long bad = ~0ull;
        KG_TRY(read_back(ctx, d_cnt.p + 2, &bad, 1));
        if (bad != ~0ull)
            return ctx_fail(ctx, KOMBGPU_EINVAL, "malformed FASTA: byte %llu (0x%02x) comes before the first record ('>' at a line start)", bad,
                            (unsigned)(unsigned char)src[bad]);
    }
    const uint32_t n_rec = (uint32_t)h_cnt[0];
    fa->n_rec = n_rec;
    fa->unterminated = n_rec && src[size - 1] != '\n';
    DevBuf<uint64_t> rec_start;
    DevBuf<uint32_t> name_len;
    KG_ALLOC(ctx, rec_start, (size_t)n_rec + 1);
    KG_ALLOC(ctx, name_len, n_rec);
    KG_CUDA(ctx, cudaMemcpyAsync(rec_start.p + n_rec, &fa->size, sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream));
    if (n_rec) KG_TRY((device_scan<uint64_t>(ctx, chunks, StartsIn{t4}, StartsOut{t4, rec_start.p}, (uint64_t *)nullptr)));

    // ---- names: lengths, hash table, duplicates (byte-compared)
    uint64_t cap = 1024;
    while (cap < 2ull * n_rec) cap <<= 1;
    int bits = 0;
    while ((1ull << bits) < cap) ++bits;
    DevBuf<unsigned long long> tab_key;
    DevBuf<uint32_t> tab_rec, slot_of, flags(ctx, 3);
    KG_ALLOC(ctx, tab_key, cap);
    KG_ALLOC(ctx, tab_rec, cap);
    KG_ALLOC(ctx, slot_of, n_rec);
    if (!flags) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
    NameTable tab{tab_key.p, tab_rec.p, (uint32_t)(cap - 1), 64 - bits};
    uint64_t seed = 0x9e3779b97f4a7c15ull;
    const uint32_t grid = grid_for(n_rec, kThreads, ctx->sm_count);
    for (int attempt = 0;; ++attempt) {
        KG_CUDA(ctx, cudaMemsetAsync(tab_key.p, 0, cap * sizeof(unsigned long long), ctx->stream));
        KG_CUDA(ctx, cudaMemsetAsync(tab_rec.p, 0xff, cap * sizeof(uint32_t), ctx->stream));
        KG_CUDA(ctx, cudaMemsetAsync(flags.p, 0xff, 3 * sizeof(uint32_t), ctx->stream));
        KG_CUDA(ctx, cudaMemsetAsync(flags.p + 1, 0, sizeof(uint32_t), ctx->stream));
        uint32_t f[3] = {kMissing, 0, kMissing};
        if (n_rec) {
            KG_LAUNCH(ctx, fasta_name_insert_kernel, grid, kThreads, 0, text.p, rec_start.p, n_rec, seed, tab, name_len.p, slot_of.p, flags.p);
            KG_LAUNCH(ctx, fasta_name_verify_kernel, grid, kThreads, 0, text.p, rec_start.p, name_len.p, n_rec, tab_rec.p, slot_of.p, flags.p);
            KG_TRY(read_back(ctx, flags.p, f, 3));
        }
        if (f[0] != kMissing) {
            uint64_t at = 0;
            KG_TRY(read_back(ctx, rec_start.p + f[0], &at, 1));
            return ctx_fail(ctx, KOMBGPU_EINVAL, "malformed FASTA: record %u (byte %llu) has an empty name", f[0], (unsigned long long)at);
        }
        if (!f[1]) {
            if (f[2] != kMissing) {
                uint64_t at = 0;
                uint32_t len = 0;
                KG_TRY(read_back(ctx, rec_start.p + f[2], &at, 1));
                KG_TRY(read_back(ctx, name_len.p + f[2], &len, 1));
                const std::string name(src + at + 1, len);
                return ctx_fail(ctx, KOMBGPU_EINVAL, "malformed FASTA: record %u repeats the name '%s' of an earlier record", f[2],
                                printable(name).c_str());
            }
            break;
        }
        if (attempt >= 3) return ctx_fail(ctx, KOMBGPU_EINTERNAL, "FASTA names: 64-bit hash collisions under four seeds");
        seed = seed * 0x9e3779b97f4a7c15ull + 0x7f4a7c15ull;
    }
    KG_CUDA(ctx, cudaEventRecord(e1, ctx->stream));
    KG_CUDA(ctx, cudaEventSynchronize(e1));
    cudaEventElapsedTime(&fa->ms_index, e0, e1);
    fa->launches += ctx->launches - launches0;
    fa->seed = seed;
    fa->cap_mask = tab.cap_mask;
    fa->shift = tab.shift;
    fa->text = text.take();
    fa->rec_start = rec_start.take();
    fa->name_len = name_len.take();
    fa->tab_key = tab_key.take();
    fa->tab_rec = tab_rec.take();
    return KOMBGPU_OK;
}

int fasta_join(kombgpu_fasta *fa, NameSpans nm, uint32_t n, uint32_t *n_missing) {
    kombgpu_ctx *ctx = fa->ctx;
    cudaEvent_t e0 = ctx->ev_a, e1 = ctx->ev_b;
    const uint64_t launches0 = ctx->launches;
    fasta_release_join(fa);
    KG_CUDA(ctx, cudaEventRecord(e0, ctx->stream));
    DevBuf<uint32_t> vrec, d_miss(ctx, 1);
    KG_ALLOC(ctx, vrec, n);
    if (!d_miss) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
    KG_CUDA(ctx, cudaMemsetAsync(d_miss.p, 0, sizeof(uint32_t), ctx->stream));
    const NameTable tab{fa->tab_key, fa->tab_rec, fa->cap_mask, fa->shift};
    if (n) KG_LAUNCH(ctx, fasta_probe_kernel, grid_for(n, kThreads, ctx->sm_count), kThreads, 0, nm, n, fa->text, fa->rec_start, fa->name_len, tab,
                     fa->seed, vrec.p, d_miss.p);
    uint32_t miss = 0;
    KG_TRY(read_back(ctx, d_miss.p, &miss, 1));
    if (miss) {   // keep the missing vertices' names: an extraction that selects one of them names it
        DevBuf<uint32_t> ids;
        DevBuf<uint64_t> off, total(ctx, 1);
        KG_ALLOC(ctx, ids, miss);
        KG_ALLOC(ctx, off, miss);
        if (!total) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
        KG_TRY((device_scan<uint32_t>(ctx, n, MissingFlagIn{vrec.p}, MissingListOut{ids.p}, (uint32_t *)nullptr)));
        KG_TRY((device_scan<uint64_t>(ctx, miss, MissingLenIn{nm, ids.p}, NoOp{}, total.p)));
        uint64_t bytes = 0;
        KG_TRY(read_back(ctx, total.p, &bytes, 1));
        DevBuf<char> names;
        KG_ALLOC(ctx, names, bytes);
        KG_TRY((device_scan<uint64_t>(ctx, miss, MissingLenIn{nm, ids.p}, MissingNameOut{nm, ids.p, off.p, names.p}, (uint64_t *)nullptr)));
        fa->missing.resize(miss);
        fa->missing_off.resize((size_t)miss + 1);
        fa->missing_names.resize(bytes);
        KG_TRY(read_back(ctx, ids.p, fa->missing.data(), miss));
        KG_TRY(read_back(ctx, off.p, fa->missing_off.data(), miss));
        if (bytes) KG_TRY(read_back(ctx, names.p, &fa->missing_names[0], bytes));
        fa->missing_off[miss] = bytes;
    }
    KG_CUDA(ctx, cudaEventRecord(e1, ctx->stream));
    KG_CUDA(ctx, cudaEventSynchronize(e1));
    cudaEventElapsedTime(&fa->ms_join, e0, e1);
    fa->launches += ctx->launches - launches0;
    fa->vrec = vrec.take();
    fa->n_vertices = n;
    fa->joined = true;
    *n_missing = miss;
    return KOMBGPU_OK;
}

int fasta_extract(kombgpu_fasta *fa, const uint8_t *mask, uint64_t *bytes) {
    kombgpu_ctx *ctx = fa->ctx;
    cudaEvent_t e0 = ctx->ev_a, e1 = ctx->ev_b;
    const uint64_t launches0 = ctx->launches;
    const uint32_t n = fa->n_vertices, n_rec = fa->n_rec;
    if (fa->out) ws_free(ctx, fa->out);
    fa->out = nullptr;
    fa->out_bytes = 0;
    fa->extracted = false;
    KG_CUDA(ctx, cudaEventRecord(e0, ctx->stream));
    DevBuf<uint8_t> d_mask, sel;
    DevBuf<uint32_t> d_err(ctx, 1);
    KG_ALLOC(ctx, d_mask, n);
    KG_ALLOC(ctx, sel, n_rec);
    if (!d_err) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
    if (n) KG_CUDA(ctx, cudaMemcpyAsync(d_mask.p, mask, n, cudaMemcpyHostToDevice, ctx->stream));
    KG_CUDA(ctx, cudaMemsetAsync(sel.p, 0, n_rec ? n_rec : 1, ctx->stream));
    KG_CUDA(ctx, cudaMemsetAsync(d_err.p, 0xff, sizeof(uint32_t), ctx->stream));
    if (n) KG_LAUNCH(ctx, fasta_mark_kernel, grid_for(n, kThreads, ctx->sm_count), kThreads, 0, d_mask.p, n, fa->vrec, sel.p, d_err.p);
    uint32_t bad = kMissing;
    KG_TRY(read_back(ctx, d_err.p, &bad, 1));
    if (bad != kMissing) {
        const size_t i = (size_t)(std::lower_bound(fa->missing.begin(), fa->missing.end(), bad) - fa->missing.begin());
        const std::string name = i < fa->missing.size() ? fa->missing_names.substr(fa->missing_off[i], fa->missing_off[i + 1] - fa->missing_off[i]) : "";
        return ctx_fail(ctx, KOMBGPU_EINVAL, "selected vertex %u (unitig '%s') has no record in the FASTA", bad, printable(name).c_str());
    }
    const uint32_t nl_rec = fa->unterminated ? n_rec - 1 : kMissing;
    DevBuf<uint64_t> out_off, first_piece, totals(ctx, 2);
    KG_ALLOC(ctx, out_off, n_rec);
    KG_ALLOC(ctx, first_piece, n_rec);
    if (!totals) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
    KG_TRY((device_scan<uint64_t>(ctx, n_rec, OutLenIn{sel.p, fa->rec_start, nl_rec}, OutOffOut{out_off.p}, totals.p)));
    KG_TRY((device_scan<uint64_t>(ctx, n_rec, PiecesIn{sel.p, fa->rec_start}, NoOp{}, totals.p + 1)));
    uint64_t tot[2] = {0, 0};
    KG_TRY(read_back(ctx, totals.p, tot, 2));
    DevBuf<char> out;
    KG_ALLOC(ctx, out, tot[0]);
    if (tot[1]) {
        DevBuf<uint32_t> piece_rec;
        KG_ALLOC(ctx, piece_rec, tot[1]);
        KG_TRY((device_scan<uint64_t>(ctx, n_rec, PiecesIn{sel.p, fa->rec_start}, PiecesOut{first_piece.p, piece_rec.p}, (uint64_t *)nullptr)));
        KG_LAUNCH(ctx, fasta_copy_kernel, grid_for(tot[1], kThreads / 32, ctx->sm_count), kThreads, 0, fa->text, fa->rec_start, out_off.p,
                  first_piece.p, piece_rec.p, tot[1], nl_rec, out.p);
    }
    KG_CUDA(ctx, cudaEventRecord(e1, ctx->stream));
    KG_CUDA(ctx, cudaEventSynchronize(e1));
    cudaEventElapsedTime(&fa->ms_extract, e0, e1);
    fa->launches += ctx->launches - launches0;
    fa->out = out.take();
    fa->out_bytes = tot[0];
    fa->extracted = true;
    *bytes = tot[0];
    return KOMBGPU_OK;
}

}  // namespace
}  // namespace kg

using namespace kg;

extern "C" {

int kombgpu_fasta_load(kombgpu_ctx *ctx, const char *text, uint64_t size, kombgpu_fasta **out) {
    if (!ctx) return KOMBGPU_EINVAL;
    if (!out || (size && !text)) return ctx_fail(ctx, KOMBGPU_EINVAL, "null argument");
    *out = nullptr;
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    kombgpu_fasta *fa = new (std::nothrow) kombgpu_fasta();
    if (!fa) return ctx_fail(ctx, KOMBGPU_ENOMEM, "host allocation");
    fa->ctx = ctx;
    const int rc = fasta_load(ctx, text, size, fa);
    if (rc != KOMBGPU_OK) {
        cudaStreamSynchronize(ctx->stream);
        fasta_release(fa);
        delete fa;
        return rc;
    }
    *out = fa;
    return KOMBGPU_OK;
}

void kombgpu_fasta_destroy(kombgpu_fasta *fa) {
    if (!fa) return;
    if (fa->ctx) cudaSetDevice(fa->ctx->device);
    fasta_release(fa);
    delete fa;
}

int kombgpu_fasta_counts(const kombgpu_fasta *fa, uint32_t *n_records, uint64_t *n_bytes) {
    if (!fa) return KOMBGPU_EINVAL;
    if (n_records) *n_records = fa->n_rec;
    if (n_bytes) *n_bytes = fa->size;
    return KOMBGPU_OK;
}

int kombgpu_fasta_join_hits(kombgpu_fasta *fa, const kombgpu_hits *names, uint32_t *n_missing) {
    if (!fa) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = fa->ctx;
    kombgpu_ctx *hctx = nullptr;
    NameSpans nm{nullptr, nullptr, nullptr};
    uint32_t n = 0;
    if (!n_missing || !names || hits_name_spans(names, &hctx, &nm.text, &nm.off, &nm.len, &n) != KOMBGPU_OK)
        return ctx_fail(ctx, KOMBGPU_EINVAL, "null argument");
    if (hctx != ctx) return ctx_fail(ctx, KOMBGPU_EINVAL, "the hits belong to another context");
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    return fasta_join(fa, nm, n, n_missing);
}

int kombgpu_fasta_join_names(kombgpu_fasta *fa, const char *bytes, const uint64_t *offsets, uint32_t n, uint32_t *n_missing) {
    if (!fa) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = fa->ctx;
    if (!n_missing || !offsets || (offsets[n] && !bytes)) return ctx_fail(ctx, KOMBGPU_EINVAL, "null argument");
    for (uint32_t v = 0; v < n; ++v)
        if (offsets[v + 1] < offsets[v] || offsets[v + 1] - offsets[v] > 0xffffffffull)
            return ctx_fail(ctx, KOMBGPU_EINVAL, "name offsets must not decrease (entry %u)", v + 1);
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    const uint64_t total = offsets[n];
    DevBuf<unsigned char> d_bytes;
    DevBuf<uint64_t> d_off;
    KG_ALLOC(ctx, d_bytes, total);
    KG_ALLOC(ctx, d_off, (size_t)n + 1);
    if (total) KG_CUDA(ctx, cudaMemcpyAsync(d_bytes.p, bytes, total, cudaMemcpyHostToDevice, ctx->stream));
    KG_CUDA(ctx, cudaMemcpyAsync(d_off.p, offsets, ((size_t)n + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream));
    const NameSpans nm{d_bytes.p, d_off.p, nullptr};
    return fasta_join(fa, nm, n, n_missing);
}

int kombgpu_fasta_extract(kombgpu_fasta *fa, const uint8_t *mask, uint32_t n, uint64_t *bytes) {
    if (!fa) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = fa->ctx;
    if (!fa->joined) return ctx_fail(ctx, KOMBGPU_ESTATE, "kombgpu_fasta_extract needs a join first");
    if (!bytes || (n && !mask)) return ctx_fail(ctx, KOMBGPU_EINVAL, "null argument");
    if (n != fa->n_vertices) return ctx_fail(ctx, KOMBGPU_EINVAL, "the mask has %u entries, the last join %u vertices", n, fa->n_vertices);
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    return fasta_extract(fa, mask, bytes);
}

int kombgpu_fasta_extract_fetch(kombgpu_fasta *fa, char *dst) {
    if (!fa) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = fa->ctx;
    if (!fa->extracted) return ctx_fail(ctx, KOMBGPU_ESTATE, "kombgpu_fasta_extract has not run");
    if (!fa->out_bytes) return KOMBGPU_OK;
    if (!dst) return ctx_fail(ctx, KOMBGPU_EINVAL, "null destination");
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    KG_CUDA(ctx, cudaMemcpyAsync(dst, fa->out, fa->out_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    KG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return KOMBGPU_OK;
}

int kombgpu_fasta_timing(const kombgpu_fasta *fa, float *ms_upload, float *ms_index, float *ms_join, float *ms_extract, uint64_t *kernel_launches) {
    if (!fa) return KOMBGPU_EINVAL;
    if (ms_upload) *ms_upload = fa->ms_upload;
    if (ms_index) *ms_index = fa->ms_index;
    if (ms_join) *ms_join = fa->ms_join;
    if (ms_extract) *ms_extract = fa->ms_extract;
    if (kernel_launches) *kernel_launches = fa->launches;
    return KOMBGPU_OK;
}

int kombgpu_anomalous(kombgpu_ctx *ctx, const double *score, uint32_t n, double whisker, double *q1, double *q3, double *fence,
                      uint32_t *n_selected, uint8_t *member) {
    if (!ctx) return KOMBGPU_EINVAL;
    if (n && !score) return ctx_fail(ctx, KOMBGPU_EINVAL, "null argument");
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    DevBuf<double> d;
    KG_ALLOC(ctx, d, n);
    if (n) KG_CUDA(ctx, cudaMemcpyAsync(d.p, score, (size_t)n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    return anomalous_dev(ctx, d.p, n, whisker, q1, q3, fence, n_selected, member);
}

int kombgpu_graph_anomalous(kombgpu_graph *g, double whisker, double *q1, double *q3, double *fence, uint32_t *n_selected, uint8_t *member) {
    if (!g) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = g->ctx;
    if (!g->has_score) return ctx_fail(ctx, KOMBGPU_ESTATE, "kombgpu_graph_anomalous needs the CORE-A scores (kombgpu_graph_corea) first");
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    const uint64_t launches0 = ctx->launches;
    const int rc = anomalous_dev(ctx, g->score, g->n, whisker, q1, q3, fence, n_selected, member);
    g->st.kernel_launches += ctx->launches - launches0;
    return rc;
}

}  // extern "C"
