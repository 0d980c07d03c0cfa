// sam.cu — SAM text -> integer hits on the device (SURVEY.md section 8, row N1).
//
// Replaces the tokenising half of Kgraph::readSAM (src/graph.cpp:197-239, at -t 1) and the thread-map merge +
// vid assignment that follows it (src/graph.cpp:242-256) for hosts that hand the raw SAM bytes to the library:
//   * a line ends at '\n'; what follows the last '\n' of a file is not processed (:206-218)
//   * lines starting with '@' are skipped (:220); "@SQ\t... SN:<name>" headers only seed the unitig numbering
//   * token 0 (QNAME) and token 2 (RNAME) under strtok("\t") rules: runs of tabs collapse (:222-231, quirk Q3)
//   * RNAME "*" is skipped (:232)
//   * read key = QNAME.substr(1, QNAME.find('/')) (:235, quirk Q2)
// Numbering (the reference's is hash order, quirk Q4; ours is the deterministic one of host/sam_tokenizer.hpp):
// read ids follow first appearance over the files in the order given; unitig ids follow @SQ header order, then
// first appearance, over unitigs with at least one hit.  Empty lines and lines with fewer than three tokens are
// undefined behaviour in the reference and are rejected (KOMBGPU_EINVAL).
//
// Kernels (all HBM-bound byte / integer work):
//   newline_count / line starts   16 bytes per thread (one uint4), SIMD byte compares; one scan writes the starts
//   parse_lines_kernel            one thread per line, touches only the head of the line (three tokens), hashes
//                                 the two spans it keeps (64 bit, seeded)
//   compaction                    one scan over the line kinds -> hit records and @SQ records in file order
//   interning                     open-addressing table keyed by the 64-bit hash (CAS insert, atomicMin of the item
//                                 index = first appearance); every item then compares its BYTES with the first
//                                 item of its slot, so equal ids mean equal strings, not equal hashes: a genuine
//                                 64-bit collision is detected and the pass repeats with another seed
//   ids                           rank of the first items (scan) = ids in order of first appearance
#include <new>
#include <vector>

#include "sam.cuh"

struct kombgpu_hits {
    kombgpu_ctx *ctx = nullptr;
    unsigned char *text = nullptr;     // every file; each starts on a 16-byte boundary, zero padded
    uint64_t text_bytes = 0;
    std::vector<uint64_t> file_base, file_size;
    uint64_t n_lines = 0, n_hits = 0;
    uint32_t n_sq = 0, n_reads = 0, n_unitigs = 0;
    uint32_t *read_key = nullptr;      // [n_hits]
    uint32_t *unitig = nullptr;        // [n_hits]
    uint64_t *name_off = nullptr;      // [n_unitigs] offset of the unitig's name in `text`
    uint32_t *name_len = nullptr;      // [n_unitigs]
    float ms_upload = 0.f, ms_parse = 0.f;
    int hash_rounds = 0;
    uint64_t launches = 0;
};

namespace kg {
namespace {

void hits_release(kombgpu_hits *h) {
    if (!h || !h->ctx) return;
    void *ptrs[] = {h->text, h->read_key, h->unitig, h->name_off, h->name_len};
    for (void *p : ptrs)
        if (p) ws_free(h->ctx, p);
    h->text = nullptr; h->read_key = nullptr; h->unitig = nullptr; h->name_off = nullptr; h->name_len = nullptr;
}

int sam_parse(kombgpu_ctx *ctx, const char *const *texts, const uint64_t *sizes, int n_files, kombgpu_hits *h) {
    cudaEvent_t e0 = ctx->ev_a, e1 = ctx->ev_b;
    const uint64_t launches0 = ctx->launches;
    // ---- upload: every file on a 16-byte boundary, zero padded (a zero byte is neither '\n' nor '\t')
    uint64_t total = 0;
    h->file_base.assign(n_files, 0);
    h->file_size.assign(sizes, sizes + n_files);
    for (int f = 0; f < n_files; ++f) {
        h->file_base[f] = total;
        total += (sizes[f] + 15) & ~15ull;
    }
    h->text_bytes = total;
    DevBuf<unsigned char> text;
    KG_ALLOC(ctx, text, total ? total : 16);
    KG_CUDA(ctx, cudaEventRecord(e0, ctx->stream));
    for (int f = 0; f < n_files; ++f) {
        if (sizes[f]) KG_CUDA(ctx, cudaMemcpyAsync(text.p + h->file_base[f], texts[f], sizes[f], cudaMemcpyHostToDevice, ctx->stream));
        const uint64_t pad = ((sizes[f] + 15) & ~15ull) - sizes[f];
        if (pad) KG_CUDA(ctx, cudaMemsetAsync(text.p + h->file_base[f] + sizes[f], 0, pad, ctx->stream));
    }
    KG_CUDA(ctx, cudaEventRecord(e1, ctx->stream));
    KG_CUDA(ctx, cudaEventSynchronize(e1));
    cudaEventElapsedTime(&h->ms_upload, e0, e1);
    KG_CUDA(ctx, cudaEventRecord(e0, ctx->stream));

    // ---- lines: count the newlines of every file, then one scan per file writes the line starts
    DevBuf<unsigned long long> d_cnt(ctx, (size_t)n_files + 1);
    if (!d_cnt) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
    KG_CUDA(ctx, cudaMemsetAsync(d_cnt.p, 0xff, sizeof(unsigned long long), ctx->stream));               // error word: min over (line << 2 | code)
    KG_CUDA(ctx, cudaMemsetAsync(d_cnt.p + 1, 0, (size_t)n_files * sizeof(unsigned long long), ctx->stream));
    for (int f = 0; f < n_files; ++f) {
        const uint64_t chunks = (sizes[f] + 15) / 16;
        if (chunks)
            KG_LAUNCH(ctx, newline_count_kernel, grid_for(chunks, kThreads * 4, ctx->sm_count), kThreads, 0,
                      reinterpret_cast<const uint4 *>(text.p + h->file_base[f]), chunks, d_cnt.p + 1 + f);
    }
    std::vector<unsigned long long> n_lines_f((size_t)n_files + 1, 0);
    KG_TRY(read_back(ctx, d_cnt.p, n_lines_f.data(), (size_t)n_files + 1));
    uint64_t n_lines = 0;
    std::vector<uint64_t> line_base(n_files, 0);
    for (int f = 0; f < n_files; ++f) { line_base[f] = n_lines; n_lines += n_lines_f[f + 1]; }
    h->n_lines = n_lines;
    // the compaction scan carries two counters in one 64-bit sum (hits low, @SQ records high) next to two status bits
    if (n_lines >= (1ull << 30)) return ctx_fail(ctx, KOMBGPU_EINVAL, "%llu lines exceed the 2^30 per-call limit", (unsigned long long)n_lines);

    DevBuf<uint8_t> kind;
    ItemBufs lkey, lname;   // per line
    KG_ALLOC(ctx, kind, n_lines);
    KG_TRY(lkey.alloc(ctx, n_lines));
    KG_TRY(lname.alloc(ctx, n_lines));
    LineTable table{kind.p, lkey.off.p, lname.off.p, lkey.hash.p, lname.hash.p, lkey.len.p, lname.len.p};
    uint64_t seed = 0x9e3779b97f4a7c15ull;
    for (int f = 0; f < n_files; ++f) {
        const uint64_t L = n_lines_f[f + 1];
        if (!L) continue;
        const uint64_t chunks = (sizes[f] + 15) / 16;
        DevBuf<uint64_t> start;
        KG_ALLOC(ctx, start, L + 1);
        KG_CUDA(ctx, cudaMemcpyAsync(start.p, &h->file_base[f], sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream));
        const uint4 *t4 = reinterpret_cast<const uint4 *>(text.p + h->file_base[f]);
        KG_TRY((device_scan<uint64_t>(ctx, chunks, NewlineIn{t4}, LineStartOut{t4, h->file_base[f], start.p}, (uint64_t *)nullptr)));
        KG_LAUNCH(ctx, parse_lines_kernel, grid_for(L, kThreads, ctx->sm_count), kThreads, 0, text.p, start.p, L, line_base[f], seed, table,
                  d_cnt.p);
    }
    unsigned long long h_err = ~0ull;
    KG_TRY(read_back(ctx, d_cnt.p, &h_err, 1));
    if (h_err != ~0ull) {
        const uint64_t line = h_err >> 2;
        int f = 0;
        while (f + 1 < n_files && line >= line_base[f + 1]) ++f;
        return ctx_fail(ctx, KOMBGPU_EINVAL, "malformed SAM (input %d, line %llu): %s", f, (unsigned long long)(line - line_base[f] + 1),
                        (h_err & 3) == 1 ? "empty line" : "line with fewer than 3 tab-separated fields");
    }

    // ---- hits and @SQ records in file order
    DevBuf<uint64_t> d_tot(ctx, 1);
    if (!d_tot) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
    ItemBufs keys, rnames, sq;
    KG_TRY(keys.alloc(ctx, n_lines));
    KG_TRY(rnames.alloc(ctx, n_lines));
    KG_TRY(sq.alloc(ctx, n_lines));
    KG_TRY((device_scan<uint64_t>(ctx, n_lines, KindIn{kind.p}, CompactLines{table, keys.view(), rnames.view(), sq.view()}, d_tot.p)));
    uint64_t tot = 0;
    KG_TRY(read_back(ctx, d_tot.p, &tot, 1));
    const uint64_t n_hits = tot & 0xffffffffull, n_sq = tot >> 32;
    h->n_hits = n_hits;
    h->n_sq = (uint32_t)n_sq;
    kind.release();
    lkey.off.release(); lkey.hash.release(); lkey.len.release();
    lname.off.release(); lname.hash.release(); lname.len.release();

    // ---- read keys: ids in order of first appearance
    DevBuf<uint32_t> key_ids, key_first;
    KG_TRY(intern_items(ctx, text.p, keys.view(), n_hits, &seed, &h->hash_rounds, key_ids, key_first, &h->n_reads));
    key_first.release();
    keys.off.release(); keys.hash.release(); keys.len.release();

    // ---- unitig names: @SQ records first, then the hits; only names with a hit become vertices
    const uint64_t n_items = n_sq + n_hits;
    ItemBufs items;
    KG_TRY(items.alloc(ctx, n_items));
    if (n_items)
        KG_LAUNCH(ctx, concat_items_kernel, grid_for(n_items, kThreads, ctx->sm_count), kThreads, 0, sq.view(), n_sq, rnames.view(), n_hits,
                  items.view());
    DevBuf<uint32_t> name_ids, name_first;
    uint32_t n_names = 0;
    KG_TRY(intern_items(ctx, text.p, items.view(), n_items, &seed, &h->hash_rounds, name_ids, name_first, &n_names));
    DevBuf<uint32_t> used, vid, d_n(ctx, 1), unitig, name_len;
    DevBuf<uint64_t> name_off;
    if (!d_n) return ctx_fail(ctx, KOMBGPU_ENOMEM, "workspace");
    KG_ALLOC(ctx, used, n_names);
    KG_ALLOC(ctx, vid, n_names);
    KG_ALLOC(ctx, unitig, n_hits);
    KG_ALLOC(ctx, name_off, n_names);
    KG_ALLOC(ctx, name_len, n_names);
    KG_CUDA(ctx, cudaMemsetAsync(used.p, 0, (size_t)(n_names ? n_names : 1) * sizeof(uint32_t), ctx->stream));
    if (n_hits) KG_LAUNCH(ctx, mark_used_kernel, grid_for(n_hits, kThreads, ctx->sm_count), kThreads, 0, name_ids.p + n_sq, n_hits, used.p);
    KG_TRY((device_scan<uint32_t>(ctx, n_names, UsedIn{used.p}, VidOut{vid.p, name_first.p, items.view(), name_off.p, name_len.p}, d_n.p)));
    if (n_hits) KG_LAUNCH(ctx, map_vid_kernel, grid_for(n_hits, kThreads, ctx->sm_count), kThreads, 0, name_ids.p + n_sq, vid.p, n_hits, unitig.p);
    KG_TRY(read_back(ctx, d_n.p, &h->n_unitigs, 1));
    KG_CUDA(ctx, cudaEventRecord(e1, ctx->stream));
    KG_CUDA(ctx, cudaEventSynchronize(e1));
    cudaEventElapsedTime(&h->ms_parse, e0, e1);
    h->launches = ctx->launches - launches0;
    h->text = text.take();
    h->read_key = key_ids.take();
    h->unitig = unitig.take();
    h->name_off = name_off.take();
    h->name_len = name_len.take();
    return KOMBGPU_OK;
}

}  // namespace

// the unitig names as spans of the device copy of the text (format.cu writes kcore.tsv from them)
int hits_name_spans(const kombgpu_hits *h, kombgpu_ctx **ctx, const unsigned char **text, const uint64_t **off, const uint32_t **len,
                    uint32_t *n_unitigs) {
    if (!h) return KOMBGPU_EINVAL;
    *ctx = h->ctx; *text = h->text; *off = h->name_off; *len = h->name_len; *n_unitigs = h->n_unitigs;
    return KOMBGPU_OK;
}

}  // namespace kg

using namespace kg;

extern "C" {

int kombgpu_sam_parse(kombgpu_ctx *ctx, const char *const *texts, const uint64_t *sizes, int n_files, kombgpu_hits **out) {
    if (!ctx) return KOMBGPU_EINVAL;
    if (!out || n_files < 0 || n_files > 64 || (n_files && (!texts || !sizes))) return ctx_fail(ctx, KOMBGPU_EINVAL, "bad argument");
    for (int f = 0; f < n_files; ++f)
        if (sizes[f] && !texts[f]) return ctx_fail(ctx, KOMBGPU_EINVAL, "null text with a non-zero size");
    *out = nullptr;
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    kombgpu_hits *h = new (std::nothrow) kombgpu_hits();
    if (!h) return ctx_fail(ctx, KOMBGPU_ENOMEM, "host allocation");
    h->ctx = ctx;
    const int rc = sam_parse(ctx, texts, sizes, n_files, h);
    if (rc != KOMBGPU_OK) {
        cudaStreamSynchronize(ctx->stream);
        hits_release(h);
        delete h;
        return rc;
    }
    *out = h;
    return KOMBGPU_OK;
}

void kombgpu_hits_destroy(kombgpu_hits *h) {
    if (!h) return;
    hits_release(h);
    delete h;
}

int kombgpu_hits_counts(const kombgpu_hits *h, uint64_t *n_hits, uint32_t *n_reads, uint32_t *n_unitigs, uint64_t *n_lines) {
    if (!h) return KOMBGPU_EINVAL;
    if (n_hits) *n_hits = h->n_hits;
    if (n_reads) *n_reads = h->n_reads;
    if (n_unitigs) *n_unitigs = h->n_unitigs;
    if (n_lines) *n_lines = h->n_lines;
    return KOMBGPU_OK;
}

int kombgpu_hits_names(const kombgpu_hits *h, uint32_t *file, uint64_t *offset, uint32_t *len) {
    if (!h) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = h->ctx;
    if (!offset || !len) return ctx_fail(ctx, KOMBGPU_EINVAL, "null argument");
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t n = h->n_unitigs;
    if (n) {
        KG_CUDA(ctx, cudaMemcpyAsync(offset, h->name_off, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
        KG_CUDA(ctx, cudaMemcpyAsync(len, h->name_len, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
        KG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    // offsets into the padded device buffer -> (input, offset inside that input)
    const int nf = (int)h->file_base.size();
    for (size_t i = 0; i < n; ++i) {
        int f = 0;
        while (f + 1 < nf && offset[i] >= h->file_base[f + 1]) ++f;
        offset[i] -= h->file_base[f];
        if (file) file[i] = (uint32_t)f;
    }
    return KOMBGPU_OK;
}

int kombgpu_hits_download(const kombgpu_hits *h, uint32_t *read_key, uint32_t *unitig) {
    if (!h) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = h->ctx;
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    if (h->n_hits) {
        if (read_key) KG_CUDA(ctx, cudaMemcpyAsync(read_key, h->read_key, h->n_hits * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
        if (unitig) KG_CUDA(ctx, cudaMemcpyAsync(unitig, h->unitig, h->n_hits * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
        KG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return KOMBGPU_OK;
}

int kombgpu_hits_device_arrays(const kombgpu_hits *h, const uint32_t **read_key, const uint32_t **unitig) {
    if (!h) return KOMBGPU_EINVAL;
    if (read_key) *read_key = h->read_key;
    if (unitig) *unitig = h->unitig;
    return KOMBGPU_OK;
}

int kombgpu_hits_timing(const kombgpu_hits *h, float *ms_upload, float *ms_parse, uint64_t *kernel_launches, int *hash_rounds) {
    if (!h) return KOMBGPU_EINVAL;
    if (ms_upload) *ms_upload = h->ms_upload;
    if (ms_parse) *ms_parse = h->ms_parse;
    if (kernel_launches) *kernel_launches = h->launches;
    if (hash_rounds) *hash_rounds = h->hash_rounds;
    return KOMBGPU_OK;
}

int kombgpu_build_graph_hits(const kombgpu_hits *h, kombgpu_graph **out) {
    if (!h) return KOMBGPU_EINVAL;
    return kombgpu_build_graph_dev(h->ctx, h->read_key, h->unitig, h->n_hits, h->n_unitigs, out);
}

}  // extern "C"
