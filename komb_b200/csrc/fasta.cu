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
// The kernels live in fasta.cuh: pfasta.cu runs them on the ranks' slices of the file.
#include <algorithm>
#include <new>
#include <string>
#include <vector>

#include "fasta.cuh"

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
    if (miss) KG_TRY(missing_to_host(ctx, nm, vrec.p, n, miss, fa->missing, fa->missing_off, fa->missing_names));
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
    char *out = nullptr;
    uint64_t total = 0;
    KG_TRY(copy_selected(ctx, fa->text, fa->rec_start, sel.p, n_rec, nl_rec, &out, &total));
    KG_CUDA(ctx, cudaEventRecord(e1, ctx->stream));
    KG_CUDA(ctx, cudaEventSynchronize(e1));
    cudaEventElapsedTime(&fa->ms_extract, e0, e1);
    fa->launches += ctx->launches - launches0;
    fa->out = out;
    fa->out_bytes = total;
    fa->extracted = true;
    *bytes = total;
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
