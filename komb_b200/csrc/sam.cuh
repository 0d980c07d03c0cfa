// sam.cuh — the kernels of SAM text -> hits (sam.cu): newline count and line starts, the per-line parse, the
// compaction of hit and @SQ records, and the string interning.  Shared by the single-GPU parse (sam.cu) and the parse
// over the ranks of a communicator (psam.cu).
#pragma once

#include "graph.cuh"
#include "primitives.cuh"
#include "strings.cuh"

namespace kg {
namespace {

enum : uint8_t { kLineSkip = 0, kLineHit = 1, kLineSq = 2 };

__device__ __forceinline__ uint32_t newlines_in(uint4 w) {
    const uint32_t nl = 0x0a0a0a0au;
    return (__popc(__vcmpeq4(w.x, nl)) + __popc(__vcmpeq4(w.y, nl)) + __popc(__vcmpeq4(w.z, nl)) + __popc(__vcmpeq4(w.w, nl))) >> 3;
}

// number of '\n' in [0, n_chunks * 16)
__global__ void __launch_bounds__(kThreads) newline_count_kernel(const uint4 *__restrict__ text, uint64_t n_chunks,
                                                                 unsigned long long *__restrict__ total) {
    uint32_t c = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_chunks; i += (uint64_t)gridDim.x * blockDim.x)
        c += newlines_in(ld_stream_u4(text + i));
    c = warp_reduce_add(c);
    if (lane_id() == 0 && c) atomicAdd(total, (unsigned long long)c);
}

struct NewlineIn {
    const uint4 *text;
    __device__ uint64_t operator()(uint64_t c) const { return newlines_in(text[c]); }
};
// start[0] is preset to the file's first byte; the k-th newline (k >= 1) at byte p gives start[k] = p + 1
struct LineStartOut {
    const uint4 *text;
    uint64_t base;        // offset of the file inside the text buffer
    uint64_t *start;
    __device__ void operator()(uint64_t c, uint64_t prefix, uint64_t cnt) const {
        if (!cnt) return;
        const uint4 w = text[c];
        const uint32_t words[4] = {w.x, w.y, w.z, w.w};
        uint64_t k = prefix;
#pragma unroll
        for (int j = 0; j < 16; ++j)
            if (((words[j >> 2] >> (8 * (j & 3))) & 0xffu) == 0x0au) start[++k] = base + c * 16 + j + 1;
    }
};

// next token of [p, end) under strtok(.., "\t") rules: leading tabs are skipped
__device__ __forceinline__ bool next_token(const unsigned char *__restrict__ t, uint64_t &p, uint64_t end, uint64_t &s, uint32_t &len) {
    while (p < end && t[p] == '\t') ++p;
    if (p >= end) return false;
    s = p;
    while (p < end && t[p] != '\t') ++p;
    len = (uint32_t)(p - s);
    return true;
}

struct LineTable {   // one record per line (global line index over all files)
    uint8_t *kind;
    uint64_t *key_off, *name_off, *key_hash, *name_hash;
    uint32_t *key_len, *name_len;
};

// one thread per line of one file; only the head of a line is read
__global__ void __launch_bounds__(kThreads) parse_lines_kernel(const unsigned char *__restrict__ text, const uint64_t *__restrict__ start,
                                                               uint64_t n_lines, uint64_t line_base, uint64_t seed, LineTable out,
                                                               unsigned long long *__restrict__ err) {
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n_lines; j += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t lo = start[j], end = start[j + 1] - 1;   // text[end] is the '\n'
        const uint64_t g = line_base + j;
        uint8_t kind = kLineSkip;
        uint64_t a_off = 0, b_off = 0;
        uint32_t a_len = 0, b_len = 0;
        if (end == lo) {
            atomicMin(err, (unsigned long long)(g << 2) | 1ull);                      // empty line
        } else if (text[lo] == '@') {
            if (end - lo > 4 && text[lo + 1] == 'S' && text[lo + 2] == 'Q' && text[lo + 3] == '\t') {
                uint64_t p = lo + 4, s = 0;
                uint32_t len = 0;
                while (next_token(text, p, end, s, len))
                    if (len > 3 && text[s] == 'S' && text[s + 1] == 'N' && text[s + 2] == ':') {
                        kind = kLineSq;
                        b_off = s + 3;
                        b_len = len - 3;
                        break;
                    }
            }
        } else {
            uint64_t p = lo, q_off = 0, skip_off = 0, r_off = 0;
            uint32_t q_len = 0, skip_len = 0, r_len = 0;
            if (!next_token(text, p, end, q_off, q_len) || !next_token(text, p, end, skip_off, skip_len) ||
                !next_token(text, p, end, r_off, r_len)) {
                atomicMin(err, (unsigned long long)(g << 2) | 2ull);                  // fewer than three fields
            } else if (!(r_len == 1 && text[r_off] == '*')) {
                // key = qname.substr(1, qname.find('/')): from index 1, as many characters as the index of the first '/'
                uint32_t slash = q_len;
                for (uint32_t i = 0; i < q_len; ++i)
                    if (text[q_off + i] == '/') { slash = i; break; }
                kind = kLineHit;
                a_off = q_off + 1;
                a_len = min(q_len - 1u, slash);
                b_off = r_off;
                b_len = r_len;
            }
        }
        out.kind[g] = kind;
        if (kind == kLineHit) {
            out.key_off[g] = a_off;
            out.key_len[g] = a_len;
            out.key_hash[g] = hash_span(text + a_off, a_len, seed);
        }
        if (kind != kLineSkip) {
            out.name_off[g] = b_off;
            out.name_len[g] = b_len;
            out.name_hash[g] = hash_span(text + b_off, b_len, seed);
        }
    }
}

struct Items {   // strings to intern: spans of the text with their hashes
    uint64_t *off, *hash;
    uint32_t *len;
};

struct KindIn {   // hits in the low word, @SQ records in the high word
    const uint8_t *kind;
    __device__ uint64_t operator()(uint64_t j) const {
        const uint8_t k = kind[j];
        return k == kLineHit ? 1ull : (k == kLineSq ? (1ull << 32) : 0ull);
    }
};
struct CompactLines {
    LineTable t;
    Items keys;    // [n_hits]
    Items rnames;  // [n_hits]
    Items sq;      // [n_sq]
    __device__ void operator()(uint64_t j, uint64_t prefix, uint64_t v) const {
        if (v == 1ull) {
            const uint32_t i = (uint32_t)prefix;
            keys.off[i] = t.key_off[j]; keys.len[i] = t.key_len[j]; keys.hash[i] = t.key_hash[j];
            rnames.off[i] = t.name_off[j]; rnames.len[i] = t.name_len[j]; rnames.hash[i] = t.name_hash[j];
        } else if (v) {
            const uint32_t i = (uint32_t)(prefix >> 32);
            sq.off[i] = t.name_off[j]; sq.len[i] = t.name_len[j]; sq.hash[i] = t.name_hash[j];
        }
    }
};

__global__ void __launch_bounds__(kThreads) concat_items_kernel(Items a, uint64_t na, Items b, uint64_t nb, Items out) {
    const uint64_t n = na + nb;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const bool first = i < na;
        const uint64_t k = first ? i : i - na;
        out.off[i] = first ? a.off[k] : b.off[k];
        out.len[i] = first ? a.len[k] : b.len[k];
        out.hash[i] = first ? a.hash[k] : b.hash[k];
    }
}

__global__ void __launch_bounds__(kThreads) rehash_kernel(const unsigned char *__restrict__ text, Items it, uint64_t n, uint64_t seed) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
        it.hash[i] = hash_span(text + it.off[i], it.len[i], seed);
}

// slot of item i = first slot, probing linearly from its home, that is empty or holds its hash; the slot remembers
// the smallest item index that landed there
__global__ void __launch_bounds__(kThreads) intern_insert_kernel(const uint64_t *__restrict__ hash, uint64_t n, unsigned long long *keys,
                                                                 uint32_t *first, uint32_t cap_mask, int shift, uint32_t *__restrict__ slot_of) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        unsigned long long h = hash[i];
        if (h == 0) h = 1;   // 0 marks an empty slot (two strings that meet here are told apart by their bytes below)
        uint32_t slot = (uint32_t)((h * 0x9e3779b97f4a7c15ull) >> shift) & cap_mask;
        while (true) {
            const unsigned long long old = atomicCAS(&keys[slot], 0ull, h);
            if (old == 0ull || old == h) break;
            slot = (slot + 1u) & cap_mask;
        }
        atomicMin(&first[slot], (uint32_t)i);
        slot_of[i] = slot;
    }
}

// equal hash must mean equal bytes: compare every item with the first item of its slot
__global__ void __launch_bounds__(kThreads) intern_verify_kernel(const unsigned char *__restrict__ text, Items it, uint64_t n,
                                                                 const uint32_t *__restrict__ first, const uint32_t *__restrict__ slot_of,
                                                                 uint32_t *__restrict__ collision) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t f = first[slot_of[i]];
        if (f == (uint32_t)i) continue;
        const uint32_t len = it.len[i];
        bool same = len == it.len[f];
        if (same) {
            const unsigned char *a = text + it.off[i], *b = text + it.off[f];
            for (uint32_t k = 0; k < len; ++k)
                if (a[k] != b[k]) { same = false; break; }
        }
        if (!same) atomicExch(collision, 1u);
    }
}

struct FirstFlagIn {
    const uint32_t *first, *slot_of;
    __device__ uint32_t operator()(uint64_t i) const { return first[slot_of[i]] == (uint32_t)i ? 1u : 0u; }
};
// the rank of a first item among the first items = the id of its string; the table's key word now holds the id
struct FirstRankOut {
    const uint32_t *slot_of;
    unsigned long long *keys;
    uint32_t *first_index;
    __device__ void operator()(uint64_t i, uint32_t prefix, uint32_t flag) const {
        if (flag) {
            keys[slot_of[i]] = prefix;
            first_index[prefix] = (uint32_t)i;
        }
    }
};
__global__ void __launch_bounds__(kThreads) intern_ids_kernel(const unsigned long long *__restrict__ keys, const uint32_t *__restrict__ slot_of,
                                                              uint64_t n, uint32_t *__restrict__ ids) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
        ids[i] = (uint32_t)keys[slot_of[i]];
}

__global__ void __launch_bounds__(kThreads) mark_used_kernel(const uint32_t *__restrict__ ids, uint64_t n, uint32_t *__restrict__ used) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) used[ids[i]] = 1u;
}
struct UsedIn {
    const uint32_t *used;
    __device__ uint32_t operator()(uint64_t d) const { return used[d]; }
};
struct VidOut {   // distinct name d with a hit becomes vertex `prefix`; its name is the span of its first item
    uint32_t *vid;
    const uint32_t *first_index;
    Items items;
    uint64_t *name_off;
    uint32_t *name_len;
    __device__ void operator()(uint64_t d, uint32_t prefix, uint32_t flag) const {
        vid[d] = prefix;
        if (flag) {
            const uint32_t f = first_index[d];
            name_off[prefix] = items.off[f];
            name_len[prefix] = items.len[f];
        }
    }
};
__global__ void __launch_bounds__(kThreads) map_vid_kernel(const uint32_t *__restrict__ ids, const uint32_t *__restrict__ vid, uint64_t n,
                                                           uint32_t *__restrict__ out) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) out[i] = vid[ids[i]];
}

struct ItemBufs {
    DevBuf<uint64_t> off, hash;
    DevBuf<uint32_t> len;
    int alloc(kombgpu_ctx *ctx, size_t n) {
        KG_ALLOC(ctx, off, n);
        KG_ALLOC(ctx, hash, n);
        KG_ALLOC(ctx, len, n);
        return KOMBGPU_OK;
    }
    Items view() { return Items{off.p, hash.p, len.p}; }
};

// ids[i] in order of first appearance, first_index[id] = first item carrying it
int intern_items(kombgpu_ctx *ctx, const unsigned char *text, Items it, uint64_t n, uint64_t *seed, int *rounds, DevBuf<uint32_t> &ids,
                 DevBuf<uint32_t> &first_index, uint32_t *n_distinct) {
    *n_distinct = 0;
    KG_ALLOC(ctx, ids, n);
    KG_ALLOC(ctx, first_index, n);
    if (n == 0) return KOMBGPU_OK;
    if (n >= 0xffffffffull) return ctx_fail(ctx, KOMBGPU_EINVAL, "more than 2^32 - 1 strings to intern");
    uint64_t cap = 1024;
    while (cap < 2 * n) cap <<= 1;
    int bits = 0;
    while ((1ull << bits) < cap) ++bits;
    DevBuf<unsigned long long> keys;
    DevBuf<uint32_t> first, slot_of, flags(ctx, 2);
    KG_ALLOC(ctx, keys, cap);
    KG_ALLOC(ctx, first, cap);
    KG_ALLOC(ctx, slot_of, n);
    if (!flags) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
    const uint32_t grid = grid_for(n, kThreads, ctx->sm_count);
    for (int attempt = 0;; ++attempt) {
        KG_CUDA(ctx, cudaMemsetAsync(keys.p, 0, cap * sizeof(unsigned long long), ctx->stream));
        KG_CUDA(ctx, cudaMemsetAsync(first.p, 0xff, cap * sizeof(uint32_t), ctx->stream));
        KG_CUDA(ctx, cudaMemsetAsync(flags.p, 0, 2 * sizeof(uint32_t), ctx->stream));
        KG_LAUNCH(ctx, intern_insert_kernel, grid, kThreads, 0, it.hash, n, keys.p, first.p, (uint32_t)(cap - 1), 64 - bits, slot_of.p);
        KG_LAUNCH(ctx, intern_verify_kernel, grid, kThreads, 0, text, it, n, first.p, slot_of.p, flags.p);
        uint32_t collision = 0;
        KG_TRY(read_back(ctx, flags.p, &collision, 1));
        ++*rounds;
        if (!collision) break;
        if (attempt >= 3) return ctx_fail(ctx, KOMBGPU_EINTERNAL, "string interning: 64-bit hash collisions under four seeds");
        *seed = *seed * 0x9e3779b97f4a7c15ull + 0x7f4a7c15ull;
        KG_LAUNCH(ctx, rehash_kernel, grid, kThreads, 0, text, it, n, *seed);
    }
    KG_TRY((device_scan<uint32_t>(ctx, n, FirstFlagIn{first.p, slot_of.p}, FirstRankOut{slot_of.p, keys.p, first_index.p}, flags.p + 1)));
    KG_LAUNCH(ctx, intern_ids_kernel, grid, kThreads, 0, keys.p, slot_of.p, n, ids.p);
    KG_TRY(read_back(ctx, flags.p + 1, n_distinct, 1));
    return KOMBGPU_OK;
}

}  // namespace
}  // namespace kg
