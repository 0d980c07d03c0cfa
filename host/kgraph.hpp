// kgraph.hpp — komb::Kgraph for the B200 path: the reference's class and method
// names (reference src/graph.h:41-63) kept as the host-side interface, every
// compute step forwarded to libkombgpu through the C ABI (include/kombgpu.h).
//
//   reference method (src/graph.cpp)          here
//   readSAM            :166-257               tokenise on the host -> integer hits + name table
//   getEdgeInfo        :259-285               nothing left to do: the mate union happens on the
//                                             device when both files' hits are sorted together
//   generateGraph      :287-393               kombgpu_build_graph (pairs, dedup, CSR)
//   readEdgeList       :395-453               writes edgelist.txt (simple edges, quirk Q7), prints
//                                             GraphInfo, calls runCore
//   runCore            :455-484               degree / coreness (kombgpu_graph_results) -> kcore.tsv
//                                             with KOMB_ONION=1 also onion.tsv (writeOnion)
//   anomalyDetection   :637-648               CORE-A scores (kombgpu_graph_results) -> CoreA_anomaly.txt
//                       (CombineCoreA::run, src/CombineCoreA.h:16-43); with KOMB_UNITIG_FASTA also the
//                                             records of the anomalous / max-truss unitigs (writeUnitigFasta; over
//                                             several GPUs each rank extracts its slice in runMulti)
// Errors follow the reference: a message on stderr and exit(EXIT_FAILURE)
// (src/graph.cpp:58-61).
#pragma once

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <future>
#include <iostream>
#include <memory>
#include <string>
#include <thread>
#include <vector>

#include "kombgpu.h"
#include "sam_tokenizer.hpp"

namespace komb {

struct HitTable {
    SamTokens tokens;                 // spans into the mapped SAM files
    std::vector<uint32_t> read_key;   // per hit
    std::vector<uint32_t> unitig;     // per hit (vid)
    std::vector<std::string> names;   // vid -> unitig name
};

// KOMB_TIMING=1: fine-grained wall-clock marks on stderr (where the drop-in's time goes outside the stage lines)
inline void timing_mark(const char *what) {
    static const bool on = getenv("KOMB_TIMING") != nullptr;
    static const auto t0 = std::chrono::steady_clock::now();
    static auto last = t0;
    if (!on) return;
    const auto now = std::chrono::steady_clock::now();
    fprintf(stderr, "[komb2 timing] %-28s +%.3f s (at %.3f s)\n", what,
            std::chrono::duration_cast<std::chrono::microseconds>(now - last).count() / 1e6,
            std::chrono::duration_cast<std::chrono::microseconds>(now - t0).count() / 1e6);
    last = now;
}

inline double seconds_since(std::chrono::steady_clock::time_point t0) {
    return std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t0).count() / 1000000.0;
}

// Page-locked host array for the large result buffers (DMA at full PCIe rate).
template <typename T>
class PinnedArray {
    kombgpu_ctx *ctx_;
    T *p_ = nullptr;
    size_t n_ = 0;

   public:
    PinnedArray(kombgpu_ctx *ctx, size_t n) : ctx_(ctx), n_(n) {
        void *q = nullptr;
        if (kombgpu_pinned_alloc(ctx, (uint64_t)(n ? n : 1) * sizeof(T), &q) != KOMBGPU_OK) {
            std::cerr << "komb2: " << kombgpu_last_error(ctx) << std::endl;
            exit(EXIT_FAILURE);
        }
        p_ = static_cast<T *>(q);
    }
    PinnedArray(const PinnedArray &) = delete;
    PinnedArray &operator=(const PinnedArray &) = delete;
    ~PinnedArray() { kombgpu_pinned_free(ctx_, p_); }
    T *data() { return p_; }
    T &operator[](size_t i) { return p_[i]; }
    size_t size() const { return n_; }
};

// ---- fast text formatting ------------------------------------------------------
inline char *put_u64(char *p, uint64_t v) {
    char tmp[24];
    int k = 0;
    do { tmp[k++] = (char)('0' + v % 10); v /= 10; } while (v);
    while (k) *p++ = tmp[--k];
    return p;
}

// format blocks of rows [lo, hi) with `fmt_block(p, lo, hi)` into per-thread buffers, then write them in order
template <typename BlockFn>
inline void write_row_blocks(FILE *f, size_t n_rows, size_t max_row_bytes, int threads, BlockFn fmt_block) {
    threads = std::max(1, threads);
    const size_t block = 1 << 16;
    std::vector<std::vector<char>> buf(threads);
    for (size_t base = 0; base < n_rows; base += block * threads) {
        std::vector<size_t> used(threads, 0);
#pragma omp parallel for num_threads(threads) schedule(static, 1)
        for (int t = 0; t < threads; ++t) {
            size_t lo = base + block * t, hi = std::min(n_rows, lo + block);
            if (lo >= hi) continue;
            buf[t].resize((hi - lo) * max_row_bytes);
            char *p = fmt_block(buf[t].data(), lo, hi);
            used[t] = (size_t)(p - buf[t].data());
        }
        for (int t = 0; t < threads; ++t)
            if (used[t]) fwrite(buf[t].data(), 1, used[t], f);
    }
}
template <typename RowFn>
inline void write_rows(FILE *f, size_t n_rows, size_t max_row_bytes, int threads, RowFn fmt_row) {
    write_row_blocks(f, n_rows, max_row_bytes, threads, [&](char *p, size_t lo, size_t hi) {
        for (size_t i = lo; i < hi; ++i) p = fmt_row(p, i);
        return p;
    });
}

class Kgraph {
    uint32_t _threads;
    uint64_t _readlength;
    kombgpu_ctx *_ctx = nullptr;
    kombgpu_graph *_graph = nullptr;
    kombgpu_hits *_hits = nullptr;       // device-resident hits when the SAM text is tokenised on the GPU
    bool _gpu_tokenise = true;           // one GPU: kombgpu_sam_parse (KOMB_TOKENIZE=host keeps the host tokeniser)
    bool _dist_tokenise = false;         // several GPUs: kombgpu_dist_sam_parse in runMulti (the same switch)
    bool _device_output = true;          // KOMB_OUTPUT=host formats the three files on the host (always without device hits:
                                         // KOMB_TOKENIZE=host)
    std::unique_ptr<PinnedArray<char>> _text[3];   // the files' bytes, formatted on the device
    uint64_t _text_bytes[3] = {0, 0, 0};
    std::vector<const MappedFile *> _sam_files;
    int _key_mode = KOMBGPU_KEY_REF32;
    int _device = 0;
    std::future<int> _ctx_ready;
    std::string _ctx_error;
    // results of the whole path, fetched in one overlapped call (kombgpu_graph_results) by readEdgeList
    std::unique_ptr<PinnedArray<uint64_t>> _efp;   // edge list in CSR form: forward offsets per source + targets
    std::unique_ptr<PinnedArray<uint32_t>> _ev;
    // multi-GPU (KOMB_GPU_DEVICES=0,1,...): one rank per device, a host thread per rank; each rank's share of the results
    struct RankOut {
        uint32_t v_lo = 0, n_local = 0;
        uint64_t n_fwd = 0;
        std::vector<uint64_t> fwd_ptr;
        std::vector<uint32_t> v;
        std::vector<int32_t> deg, core;
        std::vector<double> score;
        std::vector<std::string> names;   // unitig names of [v_lo, v_lo + n_local) (partitioned SAM parse with host output)
        uint32_t n_unitigs = 0;
        std::unique_ptr<PinnedArray<char>> text[3];   // the rank's slices of the three files, formatted on its device
        uint64_t text_bytes[3] = {0, 0, 0};
        std::unique_ptr<PinnedArray<char>> fasta;     // the rank's slice of anomalous_unitigs.fasta
        uint64_t fasta_bytes = 0;
        std::string fasta_err;            // malformed FASTA or a selected unitig without a record: reported after the three files
        bool fasta_bad_file = false;      // ... and which of the two (the message is the same on every rank)
        int rc = KOMBGPU_OK;
        std::string err;
        bool bad_input = false;           // malformed SAM: err is the parse's message, the same on every rank
    };
    std::vector<int> _devices;
    std::vector<RankOut> _ranks;         // holds page-locked text of the rank contexts: cleared before they are destroyed
    std::vector<kombgpu_ctx *> _rank_ctxs;   // one per rank, alive until the files are written (rank 0's is _ctx)
    uint64_t _m_multi = 0;
    int32_t _max_core_multi = 0;
    double _max_score_multi = 0.0;
    bool multi() const { return _devices.size() > 1; }
    void releaseRanks() {
        _ranks.clear();
        for (kombgpu_ctx *c : _rank_ctxs) kombgpu_ctx_destroy(c);
        if (!_rank_ctxs.empty()) _ctx = nullptr;
        _rank_ctxs.clear();
    }
    std::unique_ptr<PinnedArray<int32_t>> _deg, _core;
    std::unique_ptr<PinnedArray<double>> _score;
    bool _onion = false;                                    // KOMB_ONION=1: onion.tsv after kcore.tsv
    bool _fasta_anomalous = false, _fasta_truss = false;   // KOMB_UNITIG_FASTA
    std::string _fasta_path;                                // the -u FASTA
    MappedFile _fasta_file;                                 // several GPUs: mapped once, every rank reads its slice
    bool _fasta_unopened = false;                           // ... could not be mapped: reported where one GPU reports it

    // exit() must not run CUDA's teardown under a context that is still being created
    void settleDevice() { if (_ctx_ready.valid()) _ctx_ready.wait(); }
    [[noreturn]] void fileNotFoundError(const std::string &path) {
        std::cerr << "File " << path << " could not be opened. Exiting..." << std::endl;
        settleDevice();
        exit(EXIT_FAILURE);
    }
    [[noreturn]] void gpuError(const char *what, int rc) {
        std::cerr << "komb2: " << what << " failed (" << rc << "): " << kombgpu_last_error(_ctx) << std::endl;
        exit(EXIT_FAILURE);
    }

   public:
    Kgraph(uint32_t threads, uint64_t readlength, int device, int key_mode, std::vector<int> devices = {})
        : _threads(threads ? threads : 1), _readlength(readlength), _key_mode(key_mode), _device(device), _devices(std::move(devices)) {
        const char *tok_env = getenv("KOMB_TOKENIZE");
        const bool host_tok = tok_env && strcmp(tok_env, "host") == 0;
        _gpu_tokenise = !multi() && !host_tok;
        _dist_tokenise = multi() && !host_tok;
        const char *out_env = getenv("KOMB_OUTPUT");
        _device_output = (_gpu_tokenise || _dist_tokenise) && !(out_env && strcmp(out_env, "host") == 0);
        if (multi()) { timing_mark("start"); return; }   // every rank's thread creates its own context (runMulti)
        // Creating the CUDA context costs seconds on a box without the persistence daemon (1.9 - 4.1 s measured on
        // the B200 boxes, against 0.75 s for everything else on a 2.5 M-hit SAM pair): do it on a helper thread
        // while the SAM files are tokenised and interned on the host; generateGraph is the first to need it.
        timing_mark("start");
        _ctx_ready = std::async(std::launch::async, [this]() {
            int rc = kombgpu_ctx_create(_device, &_ctx);
            if (rc != KOMBGPU_OK) _ctx_error = kombgpu_last_error(nullptr);   // thread-local message: fetch it here
            return rc;
        });
        (void)_readlength;  // stored and never read, like the reference (src/graph.cpp:55)
    }
    ~Kgraph() {
        if (_ctx_ready.valid()) _ctx_ready.wait();
        _efp.reset(); _ev.reset(); _deg.reset(); _core.reset(); _score.reset();  // pinned buffers go before the context
        for (auto &t : _text) t.reset();
        releaseRanks();
        if (_graph) kombgpu_graph_destroy(_graph);
        if (_hits) kombgpu_hits_destroy(_hits);
        if (_ctx) kombgpu_ctx_destroy(_ctx);
    }

    // joins the helper thread that creates the CUDA context
    void waitForDevice() {
        if (!_ctx_ready.valid()) return;
        const int rc = _ctx_ready.get();
        timing_mark("kombgpu_ctx_create (joined)");
        if (rc != KOMBGPU_OK) {
            std::cerr << "komb2: cannot use CUDA device " << _device << ": " << _ctx_error << std::endl;
            exit(EXIT_FAILURE);
        }
    }

    // Tokenise one SAM file; the mapped file must outlive `hits` (spans point into it).
    void readSAM(const std::string &samfile, MappedFile &file, HitTable &hits, bool /*fulgor: ignored like the reference*/) {
        if (!file.open(samfile)) fileNotFoundError(samfile);
        if (_gpu_tokenise || _dist_tokenise) { _sam_files.push_back(&file); return; }   // the bytes go to the device as they are
        try {
            tokenise_sam(file, (int)_threads, hits.tokens, samfile);
        } catch (const std::exception &e) {
            std::cerr << e.what() << std::endl;
            settleDevice();
            exit(EXIT_FAILURE);
        }
    }

    // Both mates are in `hits.tokens` now: intern read keys and unitig names.  The union of the two
    // mates' unitig sets per read (reference getEdgeInfo) needs no host work: equal keys get equal ids.
    void getEdgeInfo(HitTable &hits) {
        if (_gpu_tokenise) { tokeniseOnDevice(hits); return; }
        if (_dist_tokenise) { timing_mark("map SAMs"); return; }   // every rank parses its slice of the text in runMulti
        timing_mark("tokenise SAMs");
        const size_t h = hits.tokens.keys.size();
        // ordered: ids follow first appearance, so the two mate files arrive as (at most) two runs of non-decreasing
        // read ids and the device build merges them instead of radix-sorting the hits (build.cu, merge path)
        InternResult keys = intern_spans(hits.tokens.keys, (int)_threads, true);
        hits.read_key.swap(keys.ids);
        // unitig ids: @SQ order first, then first appearance; only unitigs with a hit become vertices
        std::vector<Span> items;
        items.reserve(hits.tokens.sq.size() + h);
        items.insert(items.end(), hits.tokens.sq.begin(), hits.tokens.sq.end());
        items.insert(items.end(), hits.tokens.rnames.begin(), hits.tokens.rnames.end());
        const size_t n_sq = hits.tokens.sq.size();
        InternResult names = intern_spans(items, (int)_threads, true);
        std::vector<uint8_t> has_hit(names.n_distinct, 0);
        for (size_t i = n_sq; i < items.size(); ++i) has_hit[names.ids[i]] = 1;
        std::vector<uint32_t> vid(names.n_distinct, UINT32_MAX);
        uint32_t next = 0;
        for (uint32_t d = 0; d < names.n_distinct; ++d)
            if (has_hit[d]) {
                vid[d] = next++;
                const Span &s = items[names.first_index[d]];
                hits.names.emplace_back(s.p, s.len);
            }
        hits.unitig.resize(h);
#pragma omp parallel for num_threads(_threads) schedule(static)
        for (size_t i = 0; i < h; ++i) hits.unitig[i] = vid[names.ids[n_sq + i]];
        timing_mark("intern keys + names");
    }

    // readSAM's tokeniser and the interning of read keys and unitig names, on the device (kombgpu_sam_parse): the host
    // keeps only the unitig names, as spans of the mapped files.
    void tokeniseOnDevice(HitTable &hits) {
        timing_mark("map SAMs");
        waitForDevice();
        std::vector<const char *> texts;
        std::vector<uint64_t> sizes;
        for (const MappedFile *f : _sam_files) { texts.push_back(f->data); sizes.push_back(f->size); }
        int rc = kombgpu_sam_parse(_ctx, texts.data(), sizes.data(), (int)texts.size(), &_hits);
        if (rc == KOMBGPU_EINVAL) {   // malformed input: the host tokeniser's message and exit code
            std::cerr << kombgpu_last_error(_ctx) << std::endl;
            exit(EXIT_FAILURE);
        }
        if (rc != KOMBGPU_OK) gpuError("kombgpu_sam_parse", rc);
        uint32_t n = 0;
        kombgpu_hits_counts(_hits, nullptr, nullptr, &n, nullptr);
        if (getenv("KOMB_TIMING")) {
            float up = 0.f, parse = 0.f;
            uint64_t launches = 0;
            kombgpu_hits_timing(_hits, &up, &parse, &launches, nullptr);
            fprintf(stderr, "[komb2 timing]   device tokeniser: upload %.3f ms, parse + intern %.3f ms, %llu kernels\n", up, parse,
                    (unsigned long long)launches);
        }
        timing_mark("kombgpu_sam_parse");
        if (_device_output) return;   // kcore.tsv is formatted on the device from its copy of the text: no names on the host
        std::vector<uint32_t> file(n), len(n);
        std::vector<uint64_t> off(n);
        rc = kombgpu_hits_names(_hits, file.data(), off.data(), len.data());
        if (rc != KOMBGPU_OK) gpuError("kombgpu_hits_names", rc);
        hits.names.resize(n);
#pragma omp parallel for num_threads(_threads) schedule(static)
        for (size_t i = 0; i < (size_t)n; ++i) hits.names[i].assign(_sam_files[file[i]]->data + off[i], len[i]);
        timing_mark("unitig names to the host");
    }

    // The whole device phase over several GPUs, one host thread per rank; the ranks talk through peer memory inside
    // libkombgpu (include/kombgpu.h, peer-memory path).  By default every rank parses its slice of the mapped SAM
    // files and ends up with the hits of its own reads (kombgpu_dist_sam_parse); with KOMB_TOKENIZE=host the host's
    // hits are split by read range (a read's hits stay together) and uploaded.  By default every rank also formats
    // its slices of the three files (kombgpu_dist_graph_format) into page-locked memory of its own context; the
    // edge-list download runs under the peel and CORE-A.  The contexts live until the files are written.
    void runMulti(HitTable &hits) {
        const int world = (int)_devices.size();
        uint32_t n = (uint32_t)hits.names.size();
        const size_t h = hits.read_key.size();
        uint32_t n_reads = 0;
        for (size_t i = 0; i < h; ++i) n_reads = std::max(n_reads, hits.read_key[i] + 1);
        std::vector<const char *> texts;
        std::vector<uint64_t> sizes;
        for (const MappedFile *f : _sam_files) { texts.push_back(f->data); sizes.push_back(f->size); }
        _ranks.clear();
        _ranks.resize(world);
        void *group_slot = nullptr;
        // phase 1: the contexts (seconds each on a cold driver, so in parallel); nobody enters a collective before all exist
        std::vector<kombgpu_ctx *> ctxs(world, nullptr);
        {
            std::vector<std::thread> tc;
            for (int r = 0; r < world; ++r)
                tc.emplace_back([&, r]() {
                    const int rc = kombgpu_ctx_create(_devices[r], &ctxs[r]);
                    if (rc != KOMBGPU_OK) { _ranks[r].rc = rc; _ranks[r].err = std::string("kombgpu_ctx_create: ") + kombgpu_last_error(nullptr); }
                });
            for (auto &t : tc) t.join();
            bool ok = true;
            for (int r = 0; r < world; ++r)
                if (_ranks[r].rc != KOMBGPU_OK) {
                    std::cerr << "komb2: cannot use CUDA device " << _devices[r] << ": " << _ranks[r].err << std::endl;
                    ok = false;
                }
            if (!ok) {
                for (auto *c : ctxs) if (c) kombgpu_ctx_destroy(c);
                exit(EXIT_FAILURE);
            }
        }
        timing_mark("kombgpu_ctx_create (all devices)");
        const bool device_output = _device_output;
        const bool want_names = !device_output;   // the host writes kcore.tsv
        // anomalous_unitigs.fasta: every rank indexes its slice of the mapped -u file, joins its unitigs' names, picks
        // them by the fence over every rank's scores and extracts its slice of the output (kombgpu_dist_fasta_*)
        if (_fasta_anomalous) _fasta_unopened = !_fasta_file.open(_fasta_path);
        const bool fasta = _fasta_anomalous && !_fasta_unopened;
        std::vector<std::thread> th;
        for (int r = 0; r < world; ++r)
            th.emplace_back([&, r]() {
                RankOut &o = _ranks[r];
                kombgpu_ctx *ctx = ctxs[r];
                kombgpu_comm *comm = nullptr;
                kombgpu_dist_graph *g = nullptr;
                kombgpu_dist_hits *dh = nullptr;   // kept until kcore.tsv is formatted: the names' bytes live in it
                auto fail = [&](int rc, const char *what) {
                    o.rc = rc;
                    o.err = std::string(what) + ": " + kombgpu_last_error(ctx);
                    if (comm) kombgpu_comm_abort(comm);
                };
                // this rank's slice of one file: formatted, then downloaded on the copy stream (local, not collective)
                auto format = [&](int which) {
                    int frc = kombgpu_dist_graph_format(g, which, dh, &o.text_bytes[which]);
                    if (frc != KOMBGPU_OK) { fail(frc, "kombgpu_dist_graph_format"); return frc; }
                    o.text[which].reset(new PinnedArray<char>(ctx, o.text_bytes[which]));
                    frc = kombgpu_dist_graph_format_fetch(g, which, o.text[which]->data(), 1);
                    if (frc != KOMBGPU_OK) fail(frc, "kombgpu_dist_graph_format_fetch");
                    return frc;
                };
                int rc = kombgpu_comm_create_local(ctx, r, world, &group_slot, 0, &comm);
                if (rc != KOMBGPU_OK) fail(rc, "kombgpu_comm_create_local");
                if (rc == KOMBGPU_OK && _dist_tokenise) {
                    rc = kombgpu_dist_sam_parse(comm, texts.data(), sizes.data(), (int)texts.size(), &dh);
                    if (rc == KOMBGPU_EINVAL) { o.rc = rc; o.err = kombgpu_last_error(ctx); o.bad_input = true; }
                    else if (rc != KOMBGPU_OK) fail(rc, "kombgpu_dist_sam_parse");
                    if (rc == KOMBGPU_OK) kombgpu_dist_hits_counts(dh, nullptr, nullptr, nullptr, &o.n_unitigs, nullptr);
                    if (rc == KOMBGPU_OK && want_names) {
                        // the names of this rank's unitigs, as spans of the mapped files (kcore.tsv, the FASTA join)
                        const uint64_t step = o.n_unitigs ? ((uint64_t)o.n_unitigs + world - 1) / world : 1;
                        const uint64_t n_lo = std::min<uint64_t>(o.n_unitigs, step * r);
                        const size_t nl = (size_t)(std::min<uint64_t>(o.n_unitigs, n_lo + step) - n_lo);
                        std::vector<uint32_t> file(nl), len(nl);
                        std::vector<uint64_t> off(nl);
                        if (nl) rc = kombgpu_dist_hits_names(dh, file.data(), off.data(), len.data());   // a rank may own no unitig
                        if (rc != KOMBGPU_OK) fail(rc, "kombgpu_dist_hits_names");
                        o.names.resize(nl);
                        for (size_t i = 0; rc == KOMBGPU_OK && i < nl; ++i) o.names[i].assign(texts[file[i]] + off[i], len[i]);
                    }
                    if (rc == KOMBGPU_OK && r == 0 && getenv("KOMB_TIMING")) {
                        float up = 0.f, parse = 0.f, intern = 0.f, route = 0.f;
                        kombgpu_dist_hits_timing(dh, &up, &parse, &intern, &route, nullptr);
                        fprintf(stderr, "[komb2 timing]   rank 0 partitioned tokeniser: upload %.3f ms, parse %.3f ms, intern %.3f ms, "
                                "route %.3f ms\n", up, parse, intern, route);
                    }
                    // every rank reaches the build, which is collective: a rank whose names failed reports it there
                    if (dh) {
                        const int brc = kombgpu_dist_build_graph_hits(dh, &g);
                        if (rc == KOMBGPU_OK && brc != KOMBGPU_OK) fail(rc = brc, "kombgpu_dist_build_graph_hits");
                    }
                } else if (rc == KOMBGPU_OK) {
                    // this rank's reads: ids [lo, hi)
                    const uint32_t lo = (uint32_t)((uint64_t)n_reads * r / world), hi = (uint32_t)((uint64_t)n_reads * (r + 1) / world);
                    std::vector<uint32_t> rk, ut;
                    for (size_t i = 0; i < h; ++i)
                        if (hits.read_key[i] >= lo && hits.read_key[i] < hi) { rk.push_back(hits.read_key[i]); ut.push_back(hits.unitig[i]); }
                    rc = kombgpu_dist_build_hits(comm, rk.data(), ut.data(), rk.size(), n, &g);
                    if (rc != KOMBGPU_OK) fail(rc, "kombgpu_dist_build_hits");
                }
                if (rc == KOMBGPU_OK && device_output) rc = format(KOMBGPU_FILE_EDGELIST);   // downloads under the peel and CORE-A
                if (rc == KOMBGPU_OK && (rc = kombgpu_dist_coreness(g)) != KOMBGPU_OK) fail(rc, "kombgpu_dist_coreness");
                if (rc == KOMBGPU_OK && (rc = kombgpu_dist_corea(g, _key_mode)) != KOMBGPU_OK) fail(rc, "kombgpu_dist_corea");
                if (rc == KOMBGPU_OK) {
                    kombgpu_dist_stats st;
                    kombgpu_dist_graph_stats(g, &st);
                    o.v_lo = st.v_lo; o.n_local = st.n_local; o.n_fwd = st.n_fwd_local;
                    if (device_output) {
                        rc = format(KOMBGPU_FILE_KCORE);
                        if (rc == KOMBGPU_OK) rc = format(KOMBGPU_FILE_COREA);
                    } else {
                        o.fwd_ptr.resize((size_t)o.n_local + 1); o.v.resize(o.n_fwd);
                        o.deg.resize(o.n_local); o.core.resize(o.n_local); o.score.resize(o.n_local);
                        rc = kombgpu_dist_graph_results(g, o.deg.data(), o.core.data(), o.score.data());
                        if (rc == KOMBGPU_OK) rc = kombgpu_dist_graph_edges_csr(g, o.fwd_ptr.data(), o.v.data());
                        if (rc != KOMBGPU_OK) fail(rc, "kombgpu_dist_graph_results");
                    }
                    if (r == 0) {
                        _m_multi = st.n_edges_global;
                        kombgpu_dist_graph_summary(g, &_max_core_multi, &_max_score_multi);
                    }
                }
                if (rc == KOMBGPU_OK && fasta) rc = anomalousFastaSlice(o, ctx, comm, g, dh, hits, fail);
                if (dh) kombgpu_dist_hits_destroy(dh);
                if (g) {
                    // the downloads into the page-locked slices end before the graph's text goes
                    const int wrc = device_output ? kombgpu_dist_graph_format_wait(g) : KOMBGPU_OK;
                    if (rc == KOMBGPU_OK && wrc != KOMBGPU_OK) fail(rc = wrc, "kombgpu_dist_graph_format_wait");
                    kombgpu_dist_graph_destroy(g);
                }
                if (comm) kombgpu_comm_destroy(comm);
            });
        for (auto &t : th) t.join();
        _rank_ctxs = ctxs;   // destroyed with the ranks' page-locked text, after the three files are written
        _ctx = ctxs[0];
        if (_ranks[0].bad_input) {   // malformed SAM: the tokeniser's message (every rank has the same) and exit code
            std::cerr << _ranks[0].err << std::endl;
            exit(EXIT_FAILURE);
        }
        for (int r = 0; r < world; ++r)
            if (_ranks[r].rc != KOMBGPU_OK) {
                std::cerr << "komb2: rank " << r << " (device " << _devices[r] << "): " << _ranks[r].err << " (" << _ranks[r].rc << ")" << std::endl;
                exit(EXIT_FAILURE);
            }
        if (_dist_tokenise) {   // the ranks' name ranges, in rank order, are the names of vertices 0, 1, ...
            n = _ranks[0].n_unitigs;
            hits.names.clear();
            hits.names.reserve(n);
            for (RankOut &o : _ranks)
                for (std::string &s : o.names) hits.names.push_back(std::move(s));
        }
        timing_mark(!_dist_tokenise ? "multi-GPU build + peel + CORE-A + results"
                    : device_output ? "multi-GPU SAM parse + build + peel + CORE-A + format + download"
                                    : "multi-GPU SAM parse + build + peel + CORE-A + results");
    }

    void generateGraph(HitTable &hits) {
        if (multi()) { runMulti(hits); return; }
        waitForDevice();
        int rc = _hits ? kombgpu_build_graph_hits(_hits, &_graph)
                       : kombgpu_build_graph(_ctx, hits.read_key.data(), hits.unitig.data(), hits.read_key.size(),
                                             (uint32_t)hits.names.size(), &_graph);
        if (rc != KOMBGPU_OK) gpuError(_hits ? "kombgpu_build_graph_hits" : "kombgpu_build_graph", rc);
        timing_mark("kombgpu_build_graph");
    }

    void readEdgeList(const std::string &dir, const std::string &inputUnitigs, HitTable &hits) {
        const std::string edgelist_file = dir + "/edgelist.txt";
        FILE *ef = fopen(edgelist_file.c_str(), "w");
        if (ef == nullptr) fileNotFoundError(edgelist_file);
        auto begin_graph = std::chrono::steady_clock::now();
        uint32_t n = 0;
        uint64_t m = 0;
        if (multi()) {
            // the ranks' slices of the canonical edge list, in rank order, ARE the sorted list
            for (const RankOut &o : _ranks) n += o.n_local;
            m = _m_multi;
            for (RankOut &o : _ranks) {
                if (_device_output) {   // the slice's text, formatted on the rank's device
                    if (o.text_bytes[0] && fwrite(o.text[0]->data(), 1, o.text_bytes[0], ef) != o.text_bytes[0]) fileNotFoundError(edgelist_file);
                    o.text[0].reset();
                    continue;
                }
                const uint64_t *fp = o.fwd_ptr.data();
                write_row_blocks(ef, o.n_fwd, 24, (int)_threads, [&](char *p, size_t lo, size_t hi) {
                    size_t x = (size_t)(std::upper_bound(fp, fp + o.n_local + 1, (uint64_t)lo) - fp) - 1;
                    for (size_t i = lo; i < hi; ++i) {
                        while (fp[x + 1] <= i) ++x;
                        p = put_u64(p, (uint64_t)o.v_lo + x); *p++ = '\t';
                        p = put_u64(p, o.v[i]); *p++ = '\n';
                    }
                    return p;
                });
            }
            fclose(ef);
            timing_mark("write edgelist.txt");
            fprintf(stdout, "\nTime elapsed for initializing igraph graph: %.3f s\n", seconds_since(begin_graph));
            fprintf(stdout, "\nTime elapsed for simplifying graph: %.3f s\n", 0.0);
            fprintf(stdout, "GraphInfo...\n\tNumber of vertices: %d\n", (int)n);
            fprintf(stdout, "\tNumber of edges: %d\n", (int)m);
            FILE *uf2 = fopen(inputUnitigs.c_str(), "r");
            if (uf2 == nullptr) fileNotFoundError(inputUnitigs);
            fclose(uf2);
            auto begin_kcore2 = std::chrono::steady_clock::now();
            runCore(dir, hits);
            fprintf(stdout, "\nTime elapsed doing K-core decomposition: %.3f s\n", seconds_since(begin_kcore2));
            return;
        }
        kombgpu_graph_counts(_graph, &n, &m);
        if (_device_output) {
            // the files are formatted on the device (kombgpu_graph_format): the edge list first, its download runs on the
            // copy stream under the peel and CORE-A; the host issues one write per file
            auto fetch = [&](int which, bool async) {
                int rc = kombgpu_graph_format(_graph, which, _hits, &_text_bytes[which]);
                if (rc != KOMBGPU_OK) gpuError("kombgpu_graph_format", rc);
                _text[which].reset(new PinnedArray<char>(_ctx, _text_bytes[which]));
                rc = kombgpu_graph_format_fetch(_graph, which, _text[which]->data(), async ? 1 : 0);
                if (rc != KOMBGPU_OK) gpuError("kombgpu_graph_format_fetch", rc);
            };
            fetch(KOMBGPU_FILE_EDGELIST, true);
            int rc = kombgpu_graph_analyse(_graph, _key_mode);
            if (rc != KOMBGPU_OK) gpuError("kombgpu_graph_analyse", rc);
            fetch(KOMBGPU_FILE_KCORE, true);
            fetch(KOMBGPU_FILE_COREA, true);
            if ((rc = kombgpu_graph_format_wait(_graph)) != KOMBGPU_OK) gpuError("kombgpu_graph_format_wait", rc);
            timing_mark("format on the device + download");
            if (_text_bytes[0] && fwrite(_text[0]->data(), 1, _text_bytes[0], ef) != _text_bytes[0]) fileNotFoundError(edgelist_file);
            fclose(ef);
            _text[0].reset();
            timing_mark("write edgelist.txt");
            fprintf(stdout, "\nTime elapsed for initializing igraph graph: %.3f s\n", seconds_since(begin_graph));
            fprintf(stdout, "\nTime elapsed for simplifying graph: %.3f s\n", 0.0);
            fprintf(stdout, "GraphInfo...\n\tNumber of vertices: %d\n", (int)n);
            fprintf(stdout, "\tNumber of edges: %d\n", (int)m);
            FILE *uf3 = fopen(inputUnitigs.c_str(), "r");
            if (uf3 == nullptr) fileNotFoundError(inputUnitigs);
            fclose(uf3);
            auto begin_kcore3 = std::chrono::steady_clock::now();
            runCore(dir, hits);
            fprintf(stdout, "\nTime elapsed doing K-core decomposition: %.3f s\n", seconds_since(begin_kcore3));
            return;
        }
        // one call fetches everything the three output files need; the edge-list download (CSR form: offsets per
        // source + targets, half the bytes of two id arrays) overlaps the peel
        _efp.reset(new PinnedArray<uint64_t>(_ctx, (size_t)n + 1));
        _ev.reset(new PinnedArray<uint32_t>(_ctx, m));
        _deg.reset(new PinnedArray<int32_t>(_ctx, n));
        _core.reset(new PinnedArray<int32_t>(_ctx, n));
        _score.reset(new PinnedArray<double>(_ctx, n));
        int rc = kombgpu_graph_results_csr(_graph, _key_mode, _efp->data(), _ev->data(), _deg->data(), _core->data(), _score->data());
        if (rc != KOMBGPU_OK) gpuError("kombgpu_graph_results_csr", rc);
        timing_mark("pinned alloc + results");
        const uint64_t *fp = _efp->data();
        PinnedArray<uint32_t> &v = *_ev;
        write_row_blocks(ef, m, 24, (int)_threads, [&](char *p, size_t lo, size_t hi) {
            size_t u = (size_t)(std::upper_bound(fp, fp + n + 1, (uint64_t)lo) - fp) - 1;   // source of edge lo
            for (size_t i = lo; i < hi; ++i) {
                while (fp[u + 1] <= i) ++u;
                p = put_u64(p, u); *p++ = '\t';
                p = put_u64(p, v[i]); *p++ = '\n';
            }
            return p;
        });
        fclose(ef);
        timing_mark("write edgelist.txt");
        fprintf(stdout, "\nTime elapsed for initializing igraph graph: %.3f s\n", seconds_since(begin_graph));
        fprintf(stdout, "\nTime elapsed for simplifying graph: %.3f s\n", 0.0);  // dedup is part of the device build
        fprintf(stdout, "GraphInfo...\n\tNumber of vertices: %d\n", (int)n);
        fprintf(stdout, "\tNumber of edges: %d\n", (int)m);
        // the reference opens and parses the unitig FASTA here and discards the result
        // (src/graph.cpp:446,565-589): keep its one observable effect, the open check
        FILE *uf = fopen(inputUnitigs.c_str(), "r");
        if (uf == nullptr) fileNotFoundError(inputUnitigs);
        fclose(uf);
        auto begin_kcore = std::chrono::steady_clock::now();
        runCore(dir, hits);
        fprintf(stdout, "\nTime elapsed doing K-core decomposition: %.3f s\n", seconds_since(begin_kcore));
    }

    void runCore(const std::string &dir, HitTable &hits) {
        const std::string kcore_file = dir + "/kcore.tsv";
        const uint32_t n = (uint32_t)hits.names.size();
        if (_device_output) {
            FILE *kf = fopen(kcore_file.c_str(), "w+");
            if (kf == nullptr) fileNotFoundError(kcore_file);
            if (multi()) {   // rank 0's slice starts with the header
                for (RankOut &o : _ranks) {
                    if (o.text_bytes[1] && fwrite(o.text[1]->data(), 1, o.text_bytes[1], kf) != o.text_bytes[1]) fileNotFoundError(kcore_file);
                    o.text[1].reset();
                }
            } else {
                if (fwrite(_text[1]->data(), 1, _text_bytes[1], kf) != _text_bytes[1]) fileNotFoundError(kcore_file);
                _text[1].reset();
            }
            fclose(kf);
            timing_mark("write kcore.tsv");
            if (_onion) writeOnion(dir, hits);
            return;
        }
        // fetched by readEdgeList (one GPU) or runMulti (every rank's slice)
        std::vector<int32_t> deg_all, core_all;
        if (multi()) {
            deg_all.resize(n); core_all.resize(n);
            for (const RankOut &o : _ranks) {
                std::copy(o.deg.begin(), o.deg.end(), deg_all.begin() + o.v_lo);
                std::copy(o.core.begin(), o.core.end(), core_all.begin() + o.v_lo);
            }
        }
        const int32_t *deg = multi() ? deg_all.data() : _deg->data(), *core = multi() ? core_all.data() : _core->data();
        FILE *kcf = fopen(kcore_file.c_str(), "w+");
        if (kcf == nullptr) fileNotFoundError(kcore_file);
        fprintf(kcf, "#VID\tName\tCoreness\tDegree\n");
        size_t max_name = 0;
        for (auto &s : hits.names) max_name = std::max(max_name, s.size());
        write_rows(kcf, n, max_name + 40, (int)_threads, [&](char *p, size_t i) {
            p = put_u64(p, i); *p++ = '\t';
            memcpy(p, hits.names[i].data(), hits.names[i].size()); p += hits.names[i].size(); *p++ = '\t';
            p = put_u64(p, (uint64_t)core[i]); *p++ = '\t';
            p = put_u64(p, (uint64_t)deg[i]); *p++ = '\n';
            return p;
        });
        fclose(kcf);
        timing_mark("write kcore.tsv");
        if (_onion) writeOnion(dir, hits, core);
    }

    // <dir>/onion.tsv (KOMB_ONION=1, one GPU): the kcore.tsv row with every unitig's onion layer in the fourth column.
    // Formatted on the device with the other files, else on the host from the layers and the coreness (`core`).
    void writeOnion(const std::string &dir, const HitTable &hits, const int32_t *core = nullptr) {
        const std::string path = dir + "/onion.tsv";
        uint32_t n = 0;
        kombgpu_graph_counts(_graph, &n, nullptr);
        std::vector<uint32_t> layer(core ? n : 0);
        int rc = kombgpu_graph_onion(_graph, core ? layer.data() : nullptr, nullptr);
        if (rc != KOMBGPU_OK) gpuError("kombgpu_graph_onion", rc);
        FILE *f = fopen(path.c_str(), "w");
        if (f == nullptr) fileNotFoundError(path);
        if (!core) {
            uint64_t bytes = 0;
            if ((rc = kombgpu_graph_format(_graph, KOMBGPU_FILE_ONION, _hits, &bytes)) != KOMBGPU_OK) gpuError("kombgpu_graph_format", rc);
            PinnedArray<char> text(_ctx, bytes);
            if ((rc = kombgpu_graph_format_fetch(_graph, KOMBGPU_FILE_ONION, text.data(), 0)) != KOMBGPU_OK) gpuError("kombgpu_graph_format_fetch", rc);
            if (bytes && fwrite(text.data(), 1, bytes, f) != bytes) fileNotFoundError(path);
        } else {
            fprintf(f, "#VID\tName\tCoreness\tLayer\n");
            size_t max_name = 0;
            for (auto &s : hits.names) max_name = std::max(max_name, s.size());
            write_rows(f, n, max_name + 40, (int)_threads, [&](char *p, size_t i) {
                p = put_u64(p, i); *p++ = '\t';
                memcpy(p, hits.names[i].data(), hits.names[i].size()); p += hits.names[i].size(); *p++ = '\t';
                p = put_u64(p, (uint64_t)core[i]); *p++ = '\t';
                p = put_u64(p, layer[i]); *p++ = '\n';
                return p;
            });
        }
        fclose(f);
        timing_mark("write onion.tsv");
    }

    void anomalyDetection(const std::string &dir, bool weight, const std::string &fasta_path, const HitTable &hits) {
        uint32_t n = 0;
        int32_t max_core = 0;
        double max_score = 0.0;
        if (multi()) {
            for (const RankOut &o : _ranks) n += o.n_local;
            max_core = _max_core_multi;
            max_score = _max_score_multi;
        } else {
            kombgpu_graph_counts(_graph, &n, nullptr);
            kombgpu_graph_summary(_graph, &max_core, &max_score);
        }
        const double *score = _score ? _score->data() : nullptr;  // one GPU, host output: fetched by readEdgeList
        const double dense_ratio = (double)(max_core / 2);  // integer division, like CombineCoreA.h:24
        fprintf(stdout, "Dense Ratio: %f\n", n ? dense_ratio : 0.0);
        if (weight) {
            fprintf(stdout, "Max CoreA score: %f\n", max_score);
            const std::string anomaly_output = dir + "/CoreA_anomaly.txt";
            FILE *fp = fopen(anomaly_output.c_str(), "w+");
            if (fp == nullptr) fileNotFoundError(anomaly_output);
            if (_device_output && multi()) {
                for (const RankOut &o : _ranks)
                    if (o.text_bytes[2] && fwrite(o.text[2]->data(), 1, o.text_bytes[2], fp) != o.text_bytes[2]) fileNotFoundError(anomaly_output);
            } else if (_device_output) {
                if (_text_bytes[2] && fwrite(_text[2]->data(), 1, _text_bytes[2], fp) != _text_bytes[2]) fileNotFoundError(anomaly_output);
            } else if (multi()) {   // every rank's scores, fetched by runMulti
                for (const RankOut &o : _ranks)
                    write_rows(fp, o.n_local, 64, (int)_threads, [&](char *p, size_t i) {
                        p = put_u64(p, o.v_lo + i); *p++ = '\t';
                        p += snprintf(p, 48, "%f\n", o.score[i]);
                        return p;
                    });
            } else
            write_rows(fp, n, 64, (int)_threads, [&](char *p, size_t i) {
                p = put_u64(p, i); *p++ = '\t';
                p += snprintf(p, 48, "%f\n", score[i]);
                return p;
            });
            fclose(fp);
            timing_mark("write CoreA_anomaly.txt");
        }
        if (multi() && _fasta_anomalous) writeRankFasta(dir, fasta_path);
        else if (_fasta_anomalous || _fasta_truss) writeUnitigFasta(dir, fasta_path, hits);
        _efp.reset(); _ev.reset(); _deg.reset(); _core.reset(); _score.reset();
        for (auto &t : _text) t.reset();
        releaseRanks();
        if (_graph) kombgpu_graph_destroy(_graph);
        _graph = nullptr;
        timing_mark("free pinned + graph");
    }

    void setOnion(bool on) { _onion = on; }

    // KOMB_UNITIG_FASTA: which unitig FASTA files anomalyDetection writes, from the -u file
    void setUnitigFasta(bool anomalous, bool truss, const std::string &path) {
        _fasta_anomalous = anomalous;
        _fasta_truss = truss;
        _fasta_path = path;
    }

    // One rank's part of anomalous_unitigs.fasta (runMulti, after CORE-A; every call but the fetch is collective).  A
    // malformed file or a selected unitig without a record is kept in o.fasta_err and reported after the three files.
    template <typename Fail>
    int anomalousFastaSlice(RankOut &o, kombgpu_ctx *ctx, kombgpu_comm *comm, kombgpu_dist_graph *g, kombgpu_dist_hits *dh,
                            const HitTable &hits, Fail &fail) {
        kombgpu_dist_fasta *fa = nullptr;
        int rc = kombgpu_dist_fasta_load(comm, _fasta_file.data, _fasta_file.size, &fa);
        if (rc == KOMBGPU_EINVAL) { o.fasta_err = kombgpu_last_error(ctx); o.fasta_bad_file = true; return KOMBGPU_OK; }
        if (rc != KOMBGPU_OK) { fail(rc, "kombgpu_dist_fasta_load"); return rc; }
        uint32_t n_missing = 0;
        if (dh) {
            rc = kombgpu_dist_fasta_join_hits(fa, dh, &n_missing);
        } else {   // the host tokeniser's names of this rank's unitigs
            std::vector<uint64_t> off((size_t)o.n_local + 1, 0);
            std::string bytes;
            for (uint32_t i = 0; i < o.n_local; ++i) {
                bytes += hits.names[o.v_lo + i];
                off[i + 1] = bytes.size();
            }
            rc = kombgpu_dist_fasta_join_names(fa, bytes.data(), off.data(), o.n_local, &n_missing);
        }
        if (rc != KOMBGPU_OK) fail(rc, "kombgpu_dist_fasta_join");
        std::vector<uint8_t> mask(o.n_local, 0);
        if (rc == KOMBGPU_OK && (rc = kombgpu_dist_anomalous(g, 1.5, nullptr, nullptr, nullptr, nullptr, mask.data())) != KOMBGPU_OK)
            fail(rc, "kombgpu_dist_anomalous");
        if (rc == KOMBGPU_OK) {
            rc = kombgpu_dist_fasta_extract(fa, mask.data(), o.n_local, &o.fasta_bytes);
            if (rc == KOMBGPU_EINVAL) {
                o.fasta_err = kombgpu_last_error(ctx);
                rc = KOMBGPU_OK;
            } else if (rc != KOMBGPU_OK) {
                fail(rc, "kombgpu_dist_fasta_extract");
            } else {
                o.fasta.reset(new PinnedArray<char>(ctx, o.fasta_bytes));
                if ((rc = kombgpu_dist_fasta_extract_fetch(fa, o.fasta->data())) != KOMBGPU_OK) fail(rc, "kombgpu_dist_fasta_extract_fetch");
            }
        }
        kombgpu_dist_fasta_destroy(fa);
        return rc;
    }

    // anomalous_unitigs.fasta from several GPUs: the ranks' slices in rank order, or the error one GPU reports here
    void writeRankFasta(const std::string &dir, const std::string &fasta_path) {
        if (_fasta_unopened) fileNotFoundError(fasta_path);
        const RankOut &r0 = _ranks[0];
        if (!r0.fasta_err.empty()) {   // the same message on every rank
            std::cerr << "komb2: " << (r0.fasta_bad_file ? fasta_path : std::string("anomalous_unitigs.fasta")) << ": " << r0.fasta_err << std::endl;
            exit(EXIT_FAILURE);
        }
        const std::string path = dir + "/anomalous_unitigs.fasta";
        FILE *f = fopen(path.c_str(), "w");
        if (f == nullptr) fileNotFoundError(path);
        for (const RankOut &o : _ranks)
            if (o.fasta_bytes && fwrite(o.fasta->data(), 1, o.fasta_bytes, f) != o.fasta_bytes) fileNotFoundError(path);
        fclose(f);
        timing_mark("unitig FASTA files");
    }

    // One GPU: <dir>/anomalous_unitigs.fasta (IQR fence, whisker 1.5, on this run's CORE-A scores) and
    // <dir>/truss_unitigs.fasta (the unitigs on the edges of maximal trussness in the maximal core, the file the
    // reference's runTruss writes): the records of the -u FASTA, indexed, joined by name and copied out on the device.
    void writeUnitigFasta(const std::string &dir, const std::string &fasta_path, const HitTable &hits) {
        MappedFile file;
        if (!file.open(fasta_path)) fileNotFoundError(fasta_path);
        kombgpu_fasta *fa = nullptr;
        int rc = kombgpu_fasta_load(_ctx, file.data, file.size, &fa);
        if (rc == KOMBGPU_EINVAL) {
            std::cerr << "komb2: " << fasta_path << ": " << kombgpu_last_error(_ctx) << std::endl;
            exit(EXIT_FAILURE);
        }
        if (rc != KOMBGPU_OK) gpuError("kombgpu_fasta_load", rc);
        uint32_t n_missing = 0;
        if (_hits) {
            rc = kombgpu_fasta_join_hits(fa, _hits, &n_missing);
        } else {
            std::vector<uint64_t> off(hits.names.size() + 1, 0);
            for (size_t v = 0; v < hits.names.size(); ++v) off[v + 1] = off[v] + hits.names[v].size();
            std::string bytes;
            bytes.reserve(off.back());
            for (const std::string &nm : hits.names) bytes += nm;
            rc = kombgpu_fasta_join_names(fa, bytes.data(), off.data(), (uint32_t)hits.names.size(), &n_missing);
        }
        if (rc != KOMBGPU_OK) gpuError("kombgpu_fasta_join", rc);
        uint32_t n = 0;
        kombgpu_graph_counts(_graph, &n, nullptr);
        std::vector<uint8_t> mask(n, 0);
        auto write = [&](const char *name) {
            const std::string path = dir + "/" + name;
            uint64_t bytes = 0;
            int erc = kombgpu_fasta_extract(fa, mask.data(), n, &bytes);
            if (erc == KOMBGPU_EINVAL) {   // a selected unitig has no record: the message names it
                std::cerr << "komb2: " << name << ": " << kombgpu_last_error(_ctx) << std::endl;
                exit(EXIT_FAILURE);
            }
            if (erc != KOMBGPU_OK) gpuError("kombgpu_fasta_extract", erc);
            PinnedArray<char> buf(_ctx, bytes);
            if ((erc = kombgpu_fasta_extract_fetch(fa, buf.data())) != KOMBGPU_OK) gpuError("kombgpu_fasta_extract_fetch", erc);
            FILE *f = fopen(path.c_str(), "w");
            if (f == nullptr) fileNotFoundError(path);
            if (bytes && fwrite(buf.data(), 1, bytes, f) != bytes) fileNotFoundError(path);
            fclose(f);
        };
        if (_fasta_anomalous) {
            rc = kombgpu_graph_anomalous(_graph, 1.5, nullptr, nullptr, nullptr, nullptr, mask.data());
            if (rc != KOMBGPU_OK) gpuError("kombgpu_anomalous", rc);
            write("anomalous_unitigs.fasta");
        }
        if (_fasta_truss) {   // single GPU only (komb2.cpp refuses the combination with several GPUs)
            uint32_t n_truss = 0;
            if ((rc = kombgpu_graph_max_core_truss(_graph, nullptr, nullptr, nullptr, &n_truss)) != KOMBGPU_OK) gpuError("kombgpu_graph_max_core_truss", rc);
            std::vector<uint32_t> vids(n_truss);
            if ((rc = kombgpu_graph_truss_vertices(_graph, vids.data())) != KOMBGPU_OK) gpuError("kombgpu_graph_truss_vertices", rc);
            std::fill(mask.begin(), mask.end(), 0);
            for (uint32_t v : vids) mask[v] = 1;
            write("truss_unitigs.fasta");
        }
        kombgpu_fasta_destroy(fa);
        timing_mark("unitig FASTA files");
    }

    const kombgpu_graph *graph() const { return _graph; }
};

}  // namespace komb
