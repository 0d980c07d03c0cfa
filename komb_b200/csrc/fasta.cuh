// fasta.cuh — the kernels of the unitig FASTA (fasta.cu): record starts, names, the join probe, the extraction and the
// IQR fence.  Shared by the single-GPU calls (fasta.cu) and the calls over the ranks of a communicator (pfasta.cu).
#pragma once

#include <cstdio>
#include <string>
#include <vector>

#include "graph.cuh"
#include "primitives.cuh"
#include "strings.cuh"

namespace kg {
namespace {

constexpr uint32_t kMissing = 0xffffffffu;
constexpr uint64_t kPiece = 16384;   // bytes one warp copies at a time: long records are split into pieces of this size

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

// the name of the record whose '>' is at lo - 1 and which ends at `end`: the bytes up to the first whitespace byte
__device__ __forceinline__ uint32_t record_name_len(const unsigned char *__restrict__ text, uint64_t lo, uint64_t end) {
    uint64_t p = lo;
    while (p < end && !is_space(text[p])) ++p;
    return (uint32_t)(p - lo);
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
        const uint64_t lo = start[r] + 1;
        const uint32_t len = record_name_len(text, lo, start[r + 1]);
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

// The vertices without a record (vrec == kMissing; there are miss of them), ascending, and their names, to the host:
// an extraction that selects one of them names it.  Name i is bytes [off[i], off[i + 1]) of names.
int missing_to_host(kombgpu_ctx *ctx, NameSpans nm, const uint32_t *vrec, uint32_t n, uint32_t miss, std::vector<uint32_t> &ids_h,
                    std::vector<uint64_t> &off_h, std::string &names_h) {
    DevBuf<uint32_t> ids;
    DevBuf<uint64_t> off, total(ctx, 1);
    KG_ALLOC(ctx, ids, miss);
    KG_ALLOC(ctx, off, miss);
    if (!total) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
    KG_TRY((device_scan<uint32_t>(ctx, n, MissingFlagIn{vrec}, MissingListOut{ids.p}, (uint32_t *)nullptr)));
    KG_TRY((device_scan<uint64_t>(ctx, miss, MissingLenIn{nm, ids.p}, NoOp{}, total.p)));
    uint64_t bytes = 0;
    KG_TRY(read_back(ctx, total.p, &bytes, 1));
    DevBuf<char> names;
    KG_ALLOC(ctx, names, bytes);
    KG_TRY((device_scan<uint64_t>(ctx, miss, MissingLenIn{nm, ids.p}, MissingNameOut{nm, ids.p, off.p, names.p}, (uint64_t *)nullptr)));
    ids_h.resize(miss);
    off_h.resize((size_t)miss + 1);
    names_h.resize(bytes);
    KG_TRY(read_back(ctx, ids.p, ids_h.data(), miss));
    KG_TRY(read_back(ctx, off.p, off_h.data(), miss));
    if (bytes) KG_TRY(read_back(ctx, names.p, &names_h[0], bytes));
    off_h[miss] = bytes;
    return KOMBGPU_OK;
}

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

// The records r with sel[r] != 0 of the n_rec records at text + start[r], in order, as one text on the device (*out,
// *bytes); record nl_rec (or none: kMissing) gets a '\n' appended
int copy_selected(kombgpu_ctx *ctx, const unsigned char *text, const uint64_t *start, const uint8_t *sel, uint32_t n_rec, uint32_t nl_rec,
                  char **out_text, uint64_t *bytes) {
    DevBuf<uint64_t> out_off, first_piece, totals(ctx, 2);
    KG_ALLOC(ctx, out_off, n_rec);
    KG_ALLOC(ctx, first_piece, n_rec);
    if (!totals) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
    KG_TRY((device_scan<uint64_t>(ctx, n_rec, OutLenIn{sel, start, nl_rec}, OutOffOut{out_off.p}, totals.p)));
    KG_TRY((device_scan<uint64_t>(ctx, n_rec, PiecesIn{sel, start}, NoOp{}, totals.p + 1)));
    uint64_t tot[2] = {0, 0};
    KG_TRY(read_back(ctx, totals.p, tot, 2));
    DevBuf<char> out;
    KG_ALLOC(ctx, out, tot[0]);
    if (tot[1]) {
        DevBuf<uint32_t> piece_rec;
        KG_ALLOC(ctx, piece_rec, tot[1]);
        KG_TRY((device_scan<uint64_t>(ctx, n_rec, PiecesIn{sel, start}, PiecesOut{first_piece.p, piece_rec.p}, (uint64_t *)nullptr)));
        KG_LAUNCH(ctx, fasta_copy_kernel, grid_for(tot[1], kThreads / 32, ctx->sm_count), kThreads, 0, text, start, out_off.p,
                  first_piece.p, piece_rec.p, tot[1], nl_rec, out.p);
    }
    *out_text = out.take();
    *bytes = tot[0];
    return KOMBGPU_OK;
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

// numpy.percentile(s, 100 p, method="linear") of n sorted scores, with numpy's operations in numpy's order (the _rn
// intrinsics keep the compiler from contracting a multiply and an add into one rounding): the positions i, j of the two
// order statistics it interpolates between, and the weight t of s[j]
__device__ __forceinline__ void quartile_at(uint32_t n, double p, uint32_t *i, uint32_t *j, double *t) {
    const double h = __dsub_rn(__dmul_rn((double)n, p), p);
    const double fi = floor(h);
    *i = (uint32_t)fi;
    *j = min(*i + 1u, n - 1u);
    *t = __dsub_rn(h, fi);
}
// ... and the quartile from the order-preserving images of s[i] and s[j]
__device__ __forceinline__ double quartile_value(uint64_t ki, uint64_t kj, double t) {
    const double si = key_value(ki), sj = key_value(kj);
    const double d = __dsub_rn(sj, si);
    return t < 0.5 ? __dadd_rn(si, __dmul_rn(d, t)) : __dsub_rn(sj, __dmul_rn(d, __dsub_rn(1.0, t)));
}
// pos = {i, j} of q1 then {i, j} of q3
__device__ __forceinline__ void fence_positions(uint32_t n, uint32_t pos[4], double t[2]) {
    quartile_at(n, 0.25, &pos[0], &pos[1], &t[0]);
    quartile_at(n, 0.75, &pos[2], &pos[3], &t[1]);
}
// out = {q1, q3, fence} from the four order statistics at fence_positions (order-preserving images)
__device__ __forceinline__ void fence_from(const uint64_t stat[4], uint32_t n, double whisker, double *out) {
    uint32_t pos[4];
    double t[2];
    fence_positions(n, pos, t);
    const double q1 = quartile_value(stat[0], stat[1], t[0]), q3 = quartile_value(stat[2], stat[3], t[1]);
    out[0] = q1;
    out[1] = q3;
    out[2] = __dadd_rn(q3, __dmul_rn(whisker, __dsub_rn(q3, q1)));
}
__global__ void fence_kernel(const uint64_t *__restrict__ sorted, uint32_t n, double whisker, double *__restrict__ out) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    uint32_t pos[4];
    double t[2];
    fence_positions(n, pos, t);
    const uint64_t stat[4] = {sorted[pos[0]], sorted[pos[1]], sorted[pos[2]], sorted[pos[3]]};
    fence_from(stat, n, whisker, out);
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

std::string printable(const std::string &s) {
    std::string o;
    for (unsigned char c : s.substr(0, 200)) {
        if (c >= 0x20 && c < 0x7f) o += (char)c;
        else { char b[8]; snprintf(b, sizeof b, "\\x%02x", c); o += b; }
    }
    return s.size() > 200 ? o + "..." : o;
}

}  // namespace
}  // namespace kg
