// format.cu — the three output files formatted on the device (SURVEY.md section 8, row N2), and onion.tsv.
//
// The reference writes its files with one fprintf per row: edgelist.txt "%d\t%d\n" (src/graph.cpp:423-426),
// kcore.tsv "#VID\tName\tCoreness\tDegree\n" + "%d\t%s\t%d\t%d\n" (src/graph.cpp:467-475) and CoreA_anomaly.txt
// "%d\t%f\n" (src/CombineCoreA.h:36-39).  Here one scan computes every row's length and hands each row its offset
// in the file; the row is formatted in place by the thread that owns it, and the host receives the bytes of the file
// and issues one write.  "%f" is glibc's: six decimals of the EXACT binary value, ties to even.
#include "dgraph.cuh"
#include "primitives.cuh"

struct kombgpu_hits;
namespace kg { int hits_name_spans(const kombgpu_hits *h, kombgpu_ctx **ctx, const unsigned char **text, const uint64_t **off, const uint32_t **len,
                                   uint32_t *n_unitigs); }

namespace kg {
namespace {

constexpr char kKcoreHeader[] = "#VID\tName\tCoreness\tDegree\n";
constexpr uint64_t kKcoreHeaderLen = sizeof(kKcoreHeader) - 1;

__device__ __forceinline__ uint32_t digits_u32(uint32_t v) {
    return v < 10u ? 1u : v < 100u ? 2u : v < 1000u ? 3u : v < 10000u ? 4u : v < 100000u ? 5u : v < 1000000u ? 6u
         : v < 10000000u ? 7u : v < 100000000u ? 8u : v < 1000000000u ? 9u : 10u;
}
__device__ __forceinline__ uint32_t digits_u64(uint64_t v) {
    uint32_t d = 1;
    while (v >= 10ull) { v /= 10ull; ++d; }
    return d;
}
__device__ __forceinline__ char *put_u32(char *p, uint32_t v, uint32_t nd) {
    for (uint32_t i = nd; i > 0; --i) { p[i - 1] = (char)('0' + v % 10u); v /= 10u; }
    return p + nd;
}
__device__ __forceinline__ char *put_u64(char *p, uint64_t v, uint32_t nd) {
    for (uint32_t i = nd; i > 0; --i) { p[i - 1] = (char)('0' + (uint32_t)(v % 10ull)); v /= 10ull; }
    return p + nd;
}
// "%d" of an int32 (degrees and coreness are never negative; kept general)
__device__ __forceinline__ uint32_t digits_i32(int32_t v) { return v < 0 ? 1u + digits_u32(0u - (uint32_t)v) : digits_u32((uint32_t)v); }
__device__ __forceinline__ char *put_i32(char *p, int32_t v) {
    if (v < 0) { *p++ = '-'; return put_u32(p, 0u - (uint32_t)v, digits_u32(0u - (uint32_t)v)); }
    return put_u32(p, (uint32_t)v, digits_u32((uint32_t)v));
}

// x = m * 2^e exactly  ->  q = round_half_even(|x| * 10^6), as glibc's "%f" rounds.  |x| < 2^43 (q fits 63 bits).
// returns false for values outside that range, infinities and NaN.
__device__ __forceinline__ bool micro_units(double x, uint64_t *q_out, bool *neg) {
    const uint64_t bits = (uint64_t)__double_as_longlong(x);
    *neg = (bits >> 63) != 0;
    const uint32_t ex = (uint32_t)((bits >> 52) & 0x7ffu);
    const uint64_t man = bits & ((1ull << 52) - 1ull);
    if (ex == 0x7ffu || ex >= 1023u + 43u) return false;
    const uint64_t m = ex ? (man | (1ull << 52)) : man;
    const int s = ex ? 1075 - (int)ex : 1074;            // x = m / 2^s, s in [10, 1074] here
    const uint64_t lo = m * 1000000ull, hi = __umul64hi(m, 1000000ull);   // P = m * 10^6 < 2^73
    uint64_t q, rem_hi, rem_lo, half_hi, half_lo;
    if (s >= 128) {
        *q_out = 0;                                        // P < 2^73 <= half of 2^s: rounds to zero
        return true;
    }
    if (s >= 64) {
        const int t = s - 64;                              // 0 .. 63
        q = t ? (hi >> t) : hi;
        rem_hi = t ? (hi & ((1ull << t) - 1ull)) : 0ull;
        rem_lo = lo;
        half_hi = t ? (1ull << (t - 1)) : 0ull;
        half_lo = t ? 0ull : (1ull << 63);
    } else {
        q = (lo >> s) | (hi << (64 - s));                  // P < 2^73 and s >= 10: the quotient fits 63 bits
        rem_hi = 0;
        rem_lo = lo & ((1ull << s) - 1ull);
        half_hi = 0;
        half_lo = 1ull << (s - 1);
    }
    const bool above = rem_hi > half_hi || (rem_hi == half_hi && rem_lo > half_lo);
    const bool tie = rem_hi == half_hi && rem_lo == half_lo;
    if (above || (tie && (q & 1ull))) ++q;
    *q_out = q;
    return true;
}
__device__ __forceinline__ uint32_t f6_len(uint64_t q, bool neg) { return (neg ? 1u : 0u) + digits_u64(q / 1000000ull) + 7u; }
__device__ __forceinline__ char *put_f6(char *p, uint64_t q, bool neg) {
    if (neg) *p++ = '-';
    const uint64_t ip = q / 1000000ull;
    p = put_u64(p, ip, digits_u64(ip));
    *p++ = '.';
    return put_u32(p, (uint32_t)(q % 1000000ull), 6u);
}

// ---- edgelist.txt
struct EdgeRowLen {
    const uint64_t *edges;
    __device__ uint64_t operator()(uint64_t i) const {
        const uint64_t e = edges[i];
        return digits_u32((uint32_t)(e >> 32)) + digits_u32((uint32_t)e) + 2u;
    }
};
struct EdgeRowOut {
    const uint64_t *edges;
    char *text;
    __device__ void operator()(uint64_t i, uint64_t at, uint64_t) const {
        const uint64_t e = edges[i];
        const uint32_t u = (uint32_t)(e >> 32), v = (uint32_t)e;
        char *p = put_u32(text + at, u, digits_u32(u));
        *p++ = '\t';
        p = put_u32(p, v, digits_u32(v));
        *p = '\n';
    }
};

// ---- kcore.tsv (rows; the header is copied in front).  Row i is unitig id0 + i (id0: the first unitig of a rank's slice)
struct KcoreRowLen {
    const uint32_t *name_len;
    const int32_t *core, *deg;
    uint32_t id0;
    __device__ uint64_t operator()(uint64_t i) const {
        return digits_u32(id0 + (uint32_t)i) + name_len[i] + digits_i32(core[i]) + digits_i32(deg[i]) + 4u;
    }
};
struct KcoreRowOut {
    const unsigned char *names;
    const uint64_t *name_off;
    const uint32_t *name_len;
    const int32_t *core, *deg;
    char *text;
    uint64_t base;
    uint32_t id0;
    __device__ void operator()(uint64_t i, uint64_t at, uint64_t) const {
        const uint32_t id = id0 + (uint32_t)i;
        char *p = put_u32(text + base + at, id, digits_u32(id));
        *p++ = '\t';
        const unsigned char *nm = names + name_off[i];
        const uint32_t nl = name_len[i];
        for (uint32_t k = 0; k < nl; ++k) p[k] = (char)nm[k];
        p += nl;
        *p++ = '\t';
        p = put_i32(p, core[i]);
        *p++ = '\t';
        p = put_i32(p, deg[i]);
        *p = '\n';
    }
};

// ---- onion.tsv: the kcore.tsv row with the layer in the fourth column
constexpr char kOnionHeader[] = "#VID\tName\tCoreness\tLayer\n";
constexpr uint64_t kOnionHeaderLen = sizeof(kOnionHeader) - 1;
struct OnionRowLen {
    const uint32_t *name_len;
    const int32_t *core;
    const uint32_t *layer;
    uint32_t id0;
    __device__ uint64_t operator()(uint64_t i) const {
        return digits_u32(id0 + (uint32_t)i) + name_len[i] + digits_i32(core[i]) + digits_u32(layer[i]) + 4u;
    }
};
struct OnionRowOut {
    const unsigned char *names;
    const uint64_t *name_off;
    const uint32_t *name_len;
    const int32_t *core;
    const uint32_t *layer;
    char *text;
    uint64_t base;
    uint32_t id0;
    __device__ void operator()(uint64_t i, uint64_t at, uint64_t) const {
        const uint32_t id = id0 + (uint32_t)i;
        char *p = put_u32(text + base + at, id, digits_u32(id));
        *p++ = '\t';
        const unsigned char *nm = names + name_off[i];
        const uint32_t nl = name_len[i];
        for (uint32_t k = 0; k < nl; ++k) p[k] = (char)nm[k];
        p += nl;
        *p++ = '\t';
        p = put_i32(p, core[i]);
        *p++ = '\t';
        p = put_u32(p, layer[i], digits_u32(layer[i]));
        *p = '\n';
    }
};

// ---- CoreA_anomaly.txt (row i is unitig id0 + i)
struct ScoreRowLen {
    const double *score;
    uint32_t *err;
    uint32_t id0;
    __device__ uint64_t operator()(uint64_t i) const {
        uint64_t q = 0;
        bool neg = false;
        if (!micro_units(score[i], &q, &neg)) { atomicExch(err, 1u); q = 0; neg = false; }
        return digits_u32(id0 + (uint32_t)i) + 1u + f6_len(q, neg) + 1u;
    }
};
struct ScoreRowOut {
    const double *score;
    char *text;
    uint32_t id0;
    __device__ void operator()(uint64_t i, uint64_t at, uint64_t) const {
        uint64_t q = 0;
        bool neg = false;
        if (!micro_units(score[i], &q, &neg)) { q = 0; neg = false; }
        const uint32_t id = id0 + (uint32_t)i;
        char *p = put_u32(text + at, id, digits_u32(id));
        *p++ = '\t';
        p = put_f6(p, q, neg);
        *p = '\n';
    }
};

// two passes over the rows share one prefix: pass 1 (a scan that only sums) sizes the file, pass 2 writes it.
template <typename LenFn>
struct NoOut {
    __device__ void operator()(uint64_t, uint64_t, uint64_t) const {}
};

template <typename LenFn, typename OutFn>
int format_rows(kombgpu_ctx *ctx, uint64_t n_rows, LenFn len, OutFn (*make_out)(char *, void *), void *make_arg, uint64_t base_bytes,
                char **text_out, uint64_t *bytes_out) {
    DevBuf<uint64_t> d_total(ctx, 1);
    if (!d_total) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
    KG_TRY((device_scan<uint64_t>(ctx, n_rows, len, NoOut<LenFn>{}, d_total.p)));
    uint64_t total = 0;
    KG_TRY(read_back(ctx, d_total.p, &total, 1));
    DevBuf<char> text;
    KG_ALLOC(ctx, text, base_bytes + total);
    KG_TRY((device_scan<uint64_t>(ctx, n_rows, len, make_out(text.p, make_arg), (uint64_t *)nullptr)));
    *bytes_out = base_bytes + total;
    *text_out = text.take();
    return KOMBGPU_OK;
}

// base: bytes in front of the rows (the header, or 0 in a slice that does not start the file)
struct KcoreArgs { const unsigned char *names; const uint64_t *off; const uint32_t *len; const int32_t *core, *deg; uint64_t base; uint32_t id0; };
EdgeRowOut make_edge_out(char *text, void *arg) { return EdgeRowOut{static_cast<const uint64_t *>(arg), text}; }
KcoreRowOut make_kcore_out(char *text, void *arg) {
    const KcoreArgs *a = static_cast<const KcoreArgs *>(arg);
    return KcoreRowOut{a->names, a->off, a->len, a->core, a->deg, text, a->base, a->id0};
}
struct OnionArgs {
    const unsigned char *names;
    const uint64_t *off;
    const uint32_t *len;
    const int32_t *core;
    const uint32_t *layer;
    uint64_t base;
    uint32_t id0;
};
OnionRowOut make_onion_out(char *text, void *arg) {
    const OnionArgs *a = static_cast<const OnionArgs *>(arg);
    return OnionRowOut{a->names, a->off, a->len, a->core, a->layer, text, a->base, a->id0};
}
struct ScoreArgs { const double *score; uint32_t id0; };
ScoreRowOut make_score_out(char *text, void *arg) {
    const ScoreArgs *a = static_cast<const ScoreArgs *>(arg);
    return ScoreRowOut{a->score, text, a->id0};
}

// the rows of unitigs id0 .. id0 + n - 1
int format_scores(kombgpu_ctx *ctx, const double *score_dev, uint32_t n, uint32_t id0, char **text, uint64_t *bytes) {
    DevBuf<uint32_t> err(ctx, 1);
    if (!err) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
    KG_CUDA(ctx, cudaMemsetAsync(err.p, 0, sizeof(uint32_t), ctx->stream));
    ScoreArgs a{score_dev, id0};
    KG_TRY(format_rows(ctx, n, ScoreRowLen{score_dev, err.p, id0}, make_score_out, &a, 0, text, bytes));
    uint32_t h_err = 0;
    KG_TRY(read_back(ctx, err.p, &h_err, 1));
    if (h_err) {
        ws_free(ctx, *text);
        *text = nullptr;
        return ctx_fail(ctx, KOMBGPU_EINVAL, "a score is not finite or not below 2^43: outside the device formatter's range");
    }
    return KOMBGPU_OK;
}

// the text of file `which` to the host: async != 0 on the copy stream, behind everything the compute stream has queued
int fetch_text(kombgpu_ctx *ctx, const char *text, uint64_t bytes, char *dst, int async) {
    if (!dst && bytes) return ctx_fail(ctx, KOMBGPU_EINVAL, "null destination");
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    if (!bytes) return KOMBGPU_OK;
    if (async) {
        // later compute on the stream overlaps the download
        cudaEvent_t ev = nullptr;
        KG_CUDA(ctx, cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        cudaError_t e = cudaEventRecord(ev, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->copy_stream, ev, 0);
        if (e == cudaSuccess) e = cudaMemcpyAsync(dst, text, bytes, cudaMemcpyDeviceToHost, ctx->copy_stream);
        cudaEventDestroy(ev);
        KG_CUDA(ctx, e);
        return KOMBGPU_OK;
    }
    KG_CUDA(ctx, cudaMemcpyAsync(dst, text, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    KG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return KOMBGPU_OK;
}

void release_texts(kombgpu_ctx *ctx, char **text, uint64_t *text_bytes, int n_files) {
    for (int w = 0; w < n_files; ++w) {
        if (text[w]) ws_free(ctx, text[w]);
        text[w] = nullptr;
        text_bytes[w] = 0;
    }
}

}  // namespace

void format_release(kombgpu_graph *g) { release_texts(g->ctx, g->text, g->text_bytes, 4); }
void dist_format_release(kombgpu_dist_graph *g) { release_texts(g->ctx, g->text, g->text_bytes, 4); }

}  // namespace kg

using namespace kg;

extern "C" {

int kombgpu_graph_format(kombgpu_graph *g, int which, const kombgpu_hits *names, uint64_t *bytes) {
    if (!g) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = g->ctx;
    if (!bytes || which < 0 || which > KOMBGPU_FILE_ONION) return ctx_fail(ctx, KOMBGPU_EINVAL, "bad argument");
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    if (g->text[which]) { *bytes = g->text_bytes[which]; return KOMBGPU_OK; }
    const uint64_t launches0 = ctx->launches;
    char *text = nullptr;
    uint64_t total = 0;
    if (which == KOMBGPU_FILE_EDGELIST) {
        if (g->n_edges && !g->edges) return ctx_fail(ctx, KOMBGPU_ESTATE, "the graph was adopted from a CSR: no canonical edge list");
        KG_TRY(format_rows(ctx, g->n_edges, EdgeRowLen{g->edges}, make_edge_out, (void *)g->edges, 0, &text, &total));
    } else if (which == KOMBGPU_FILE_KCORE) {
        if (!g->has_core) return ctx_fail(ctx, KOMBGPU_ESTATE, "kombgpu_coreness has not run");
        kombgpu_ctx *hctx = nullptr;
        KcoreArgs a{};
        uint32_t n_names = 0;
        if (!names || hits_name_spans(names, &hctx, &a.names, &a.off, &a.len, &n_names) != KOMBGPU_OK || hctx != ctx || n_names != g->n)
            return ctx_fail(ctx, KOMBGPU_EINVAL, "kcore.tsv needs the unitig names: the kombgpu_hits this graph was built from");
        a.core = g->core;
        a.deg = g->deg;
        a.base = kKcoreHeaderLen;
        KG_TRY(format_rows(ctx, g->n, KcoreRowLen{a.len, a.core, a.deg, 0u}, make_kcore_out, &a, kKcoreHeaderLen, &text, &total));
        KG_CUDA(ctx, cudaMemcpyAsync(text, kKcoreHeader, kKcoreHeaderLen, cudaMemcpyHostToDevice, ctx->stream));
    } else if (which == KOMBGPU_FILE_ONION) {
        if (!g->has_onion) return ctx_fail(ctx, KOMBGPU_ESTATE, "kombgpu_graph_onion has not run");
        kombgpu_ctx *hctx = nullptr;
        OnionArgs a{};
        uint32_t n_names = 0;
        if (!names || hits_name_spans(names, &hctx, &a.names, &a.off, &a.len, &n_names) != KOMBGPU_OK || hctx != ctx || n_names != g->n)
            return ctx_fail(ctx, KOMBGPU_EINVAL, "onion.tsv needs the unitig names: the kombgpu_hits this graph was built from");
        a.core = g->onion_core;
        a.layer = g->onion_layer;
        a.base = kOnionHeaderLen;
        KG_TRY(format_rows(ctx, g->n, OnionRowLen{a.len, a.core, a.layer, 0u}, make_onion_out, &a, kOnionHeaderLen, &text, &total));
        KG_CUDA(ctx, cudaMemcpyAsync(text, kOnionHeader, kOnionHeaderLen, cudaMemcpyHostToDevice, ctx->stream));
    } else {
        if (!g->has_score) return ctx_fail(ctx, KOMBGPU_ESTATE, "kombgpu_graph_corea has not run");
        KG_TRY(format_scores(ctx, g->score, g->n, 0u, &text, &total));
    }
    g->text[which] = text;
    g->text_bytes[which] = total;
    g->st.kernel_launches += ctx->launches - launches0;
    *bytes = total;
    return KOMBGPU_OK;
}

int kombgpu_graph_format_fetch(kombgpu_graph *g, int which, char *dst, int async) {
    if (!g) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = g->ctx;
    if (which < 0 || which > KOMBGPU_FILE_ONION || !g->text[which]) return ctx_fail(ctx, KOMBGPU_ESTATE, "kombgpu_graph_format has not run for this file");
    return fetch_text(ctx, g->text[which], g->text_bytes[which], dst, async);
}

int kombgpu_graph_format_wait(kombgpu_graph *g) {
    if (!g) return KOMBGPU_EINVAL;
    KG_CUDA(g->ctx, cudaSetDevice(g->ctx->device));
    KG_CUDA(g->ctx, cudaStreamSynchronize(g->ctx->copy_stream));
    return KOMBGPU_OK;
}

int kombgpu_format_corea(kombgpu_ctx *ctx, const double *score, uint32_t n, char *dst, uint64_t capacity, uint64_t *bytes) {
    if (!ctx) return KOMBGPU_EINVAL;
    if (!bytes || (n && !score)) return ctx_fail(ctx, KOMBGPU_EINVAL, "null argument");
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    DevBuf<double> d;
    KG_ALLOC(ctx, d, n);
    if (n) KG_CUDA(ctx, cudaMemcpyAsync(d.p, score, (size_t)n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    char *text = nullptr;
    uint64_t total = 0;
    KG_TRY(format_scores(ctx, d.p, n, 0u, &text, &total));
    DevBuf<char> hold;
    hold.ctx = ctx;
    hold.p = text;
    *bytes = total;
    if (total > capacity || (total && !dst)) return ctx_fail(ctx, KOMBGPU_EINVAL, "the text takes %llu bytes, the buffer holds %llu", (unsigned long long)total, (unsigned long long)capacity);
    if (total) {
        KG_CUDA(ctx, cudaMemcpyAsync(dst, text, total, cudaMemcpyDeviceToHost, ctx->stream));
        KG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return KOMBGPU_OK;
}

// ---- the partitioned graph: this rank's slice of each file (local, not collective)

int kombgpu_dist_graph_format(kombgpu_dist_graph *g, int which, const kombgpu_dist_hits *names, uint64_t *bytes) {
    if (!g) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = g->ctx;
    if (!bytes || which < 0 || which > KOMBGPU_FILE_ONION) return ctx_fail(ctx, KOMBGPU_EINVAL, "bad argument");
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    if (g->text[which]) { *bytes = g->text_bytes[which]; return KOMBGPU_OK; }
    char *text = nullptr;
    uint64_t total = 0;
    if (which == KOMBGPU_FILE_EDGELIST) {
        KG_TRY(format_rows(ctx, g->n_fwd, EdgeRowLen{g->edges}, make_edge_out, (void *)g->edges, 0, &text, &total));
    } else if (which == KOMBGPU_FILE_KCORE) {
        if (!g->has_core) return ctx_fail(ctx, KOMBGPU_ESTATE, "kombgpu_dist_coreness has not run");
        DistNames nm{};
        if (!names || dist_hits_name_text(names, &nm) != KOMBGPU_OK || nm.comm != g->comm || nm.n_unitigs != g->n_global || nm.v_lo != g->v_lo ||
            nm.n_local != g->n_local)
            return ctx_fail(ctx, KOMBGPU_EINVAL, "kcore.tsv needs the unitig names: the kombgpu_dist_hits this graph was built from");
        // the header starts rank 0's slice, the file's first (even when the graph is empty)
        const uint64_t head = g->comm->rank == 0 ? kKcoreHeaderLen : 0;
        KcoreArgs a{nm.bytes, nm.off, nm.len, g->core, g->deg, head, g->v_lo};
        KG_TRY(format_rows(ctx, g->n_local, KcoreRowLen{a.len, a.core, a.deg, g->v_lo}, make_kcore_out, &a, head, &text, &total));
        if (head) KG_CUDA(ctx, cudaMemcpyAsync(text, kKcoreHeader, kKcoreHeaderLen, cudaMemcpyHostToDevice, ctx->stream));
    } else if (which == KOMBGPU_FILE_ONION) {
        // the names are checked before the state: a call without the graph's own names is wrong whenever it comes
        DistNames nm{};
        if (!names || dist_hits_name_text(names, &nm) != KOMBGPU_OK || nm.comm != g->comm || nm.n_unitigs != g->n_global || nm.v_lo != g->v_lo ||
            nm.n_local != g->n_local)
            return ctx_fail(ctx, KOMBGPU_EINVAL, "onion.tsv needs the unitig names: the kombgpu_dist_hits this graph was built from");
        if (!g->has_onion) return ctx_fail(ctx, KOMBGPU_ESTATE, "kombgpu_dist_onion has not run");
        const uint64_t head = g->comm->rank == 0 ? kOnionHeaderLen : 0;
        OnionArgs a{nm.bytes, nm.off, nm.len, g->onion_core, g->onion_layer, head, g->v_lo};
        KG_TRY(format_rows(ctx, g->n_local, OnionRowLen{a.len, a.core, a.layer, g->v_lo}, make_onion_out, &a, head, &text, &total));
        if (head) KG_CUDA(ctx, cudaMemcpyAsync(text, kOnionHeader, kOnionHeaderLen, cudaMemcpyHostToDevice, ctx->stream));
    } else {
        if (!g->has_score) return ctx_fail(ctx, KOMBGPU_ESTATE, "kombgpu_dist_corea has not run");
        KG_TRY(format_scores(ctx, g->score, g->n_local, g->v_lo, &text, &total));
    }
    g->text[which] = text;
    g->text_bytes[which] = total;
    *bytes = total;
    return KOMBGPU_OK;
}

int kombgpu_dist_graph_format_fetch(kombgpu_dist_graph *g, int which, char *dst, int async) {
    if (!g) return KOMBGPU_EINVAL;
    if (which < 0 || which > KOMBGPU_FILE_ONION || !g->text[which]) return ctx_fail(g->ctx, KOMBGPU_ESTATE, "kombgpu_dist_graph_format has not run for this file");
    return fetch_text(g->ctx, g->text[which], g->text_bytes[which], dst, async);
}

int kombgpu_dist_graph_format_wait(kombgpu_dist_graph *g) {
    if (!g) return KOMBGPU_EINVAL;
    KG_CUDA(g->ctx, cudaSetDevice(g->ctx->device));
    KG_CUDA(g->ctx, cudaStreamSynchronize(g->ctx->copy_stream));
    return KOMBGPU_OK;
}

}  // extern "C"
