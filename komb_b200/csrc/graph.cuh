// graph.cuh — the device-resident unitig graph and the stage entry points that
// the C ABI (capi.cu) strings together.
#pragma once

#include "common.cuh"

namespace kg {
// the maximal core and the trussness of its edges (truss.cu), computed on demand
struct MaxCoreTruss {
    uint32_t n_core = 0, n_vertices = 0;
    uint64_t m = 0;
    int32_t tmax = 0;
    uint32_t *core_vid = nullptr;   // [n_core] original ids of the maximal core, ascending
    uint64_t *edges = nullptr;      // [m] induced edges, compact ids (a << 32 | b), canonical order
    int32_t *truss = nullptr;       // [m]
    uint32_t *vertices = nullptr;   // [n_vertices] original ids of the unitigs on edges of maximal trussness
};
}  // namespace kg

struct kombgpu_graph {
    kombgpu_ctx *ctx = nullptr;
    uint32_t n = 0;            // vertices (hit unitigs)
    uint64_t n_edges = 0;      // simple undirected edges
    uint64_t *edges = nullptr;   // [E]   packed (u << 32 | v), u < v, ascending
    uint64_t *row_ptr = nullptr; // [n+1] CSR offsets of the symmetric graph
    uint32_t *col = nullptr;     // [2E]  neighbours, every row ascending
    uint32_t *fwd_start = nullptr; // [n+1] forward index of the edge list: edges [fwd_start[u], fwd_start[u+1]) have source u
    uint32_t *mult = nullptr;    // [E]   pairs (reads, or input duplicates) that support each edge
    uint32_t build_chunks = 0;   // chunks the pairs were reduced in (1: one shot; 0: adopted from a CSR)
    int32_t *deg = nullptr;      // [n]
    int32_t *core = nullptr;     // [n]   after peel
    double *score = nullptr;     // [n]   after CORE-A
    double max_score = 0.0;
    bool has_core = false, has_score = false;
    kombgpu_stats st{};
    bool has_truss = false;
    kg::MaxCoreTruss tr;
    // output files formatted on the device (format.cu): edgelist.txt, kcore.tsv, CoreA_anomaly.txt
    char *text[3] = {nullptr, nullptr, nullptr};
    uint64_t text_bytes[3] = {0, 0, 0};
};

namespace kg {

// stage 1 (build.cu) — inputs are device pointers
int build_from_hits(kombgpu_ctx *ctx, const uint32_t *read_key, const uint32_t *unitig, uint64_t n_hits,
                    uint32_t n_vertices, kombgpu_graph *g);
int build_from_pairs(kombgpu_ctx *ctx, const uint32_t *u, const uint32_t *v, uint64_t n_pairs, uint32_t n_vertices,
                     kombgpu_graph *g);

// building blocks of stage 1 shared with the partitioned (multi-GPU) path (build.cu)
// `mult` (optional): receives, per unique edge, how many emitted pairs collapsed into it
// Any number of pairs: from 2^32 on (or above KOMBGPU_PAIR_CHUNK) they are reduced in chunks; `n_chunks` (optional)
// receives how many (1 for the one-shot path).
int hits_to_edges(kombgpu_ctx *ctx, const uint32_t *read_key, const uint32_t *unitig, uint64_t n_hits, uint32_t n_vertices,
                  DevBuf<uint64_t> &edges, uint64_t *n_edges, kombgpu_stats *st, DevBuf<uint32_t> *mult = nullptr,
                  uint32_t *n_chunks = nullptr);
int pairs_to_edges(kombgpu_ctx *ctx, const uint32_t *u, const uint32_t *v, uint64_t n_pairs, uint32_t n_vertices,
                   DevBuf<uint64_t> &edges, uint64_t *n_edges, DevBuf<uint32_t> *mult = nullptr, uint32_t *n_chunks = nullptr);
// Steps 1-2 of a build from hits: the unique hits grouped by read, the reads with >= 2 unitigs as segments and the
// global index of every segment's first pair.  P is known before any pair exists; emit(p0, p1, dst) then writes the
// canonical keys (min << 32 | max) of pairs [p0, p1) to dst[0, p1 - p0), in emission order (not sorted, duplicates in):
// the whole list in one shot or one chunk of it (a chunk may start inside a read's clique).
struct HitPairs {
    kombgpu_ctx *ctx = nullptr;
    DevBuf<uint64_t> ha, hb, hc, seg_base;
    DevBuf<uint32_t> seg_head, seg_tail, tile_seg;
    const uint64_t *hits = nullptr;   // unique hits grouped by read, inside ha / hb / hc
    uint32_t n_seg = 0;
    uint64_t n_pairs = 0;
    int emit(uint64_t p0, uint64_t p1, uint64_t *dst);
    void release();
};
int count_hit_pairs(kombgpu_ctx *ctx, const uint32_t *read_key, const uint32_t *unitig, uint64_t n_hits, uint32_t n_vertices,
                    HitPairs *hp, kombgpu_stats *st);
// (u, v) pairs -> canonical keys (min << 32 | max) in dst[0, n), input order; KOMBGPU_EINVAL when an id is >= n_vertices
int pack_pairs(kombgpu_ctx *ctx, const uint32_t *u, const uint32_t *v, uint64_t n, uint32_t n_vertices, uint64_t *dst);

// Pairs reduced a chunk at a time (build.cu, "chunked path"): the chunk size, and KOMBGPU_PAIR_CHUNK (0 when unset)
constexpr uint64_t kPairChunk = (1ull << 30) - (1ull << 20);   // bounds the memory of a chunk: its keys, sort buffer, counts
uint64_t pair_chunk_env();
// the running edge list of a chunked build: sorted unique keys and how many pairs support each (saturating at 2^32 - 1)
struct EdgeRun {
    DevBuf<uint64_t> keys;
    DevBuf<uint32_t> cnt;
    uint64_t n = 0;
};
// one sorted chunk of pair keys (duplicates and loops in, n_c < 2^32) -> sorted unique (key, count) in cuniq / ccnt
// (n_c entries of room each), merged into the running list.  KOMBGPU_EINVAL when the list would reach 2^32 edges.
int merge_sorted_chunk(kombgpu_ctx *ctx, const uint64_t *sorted, uint64_t n_c, uint64_t *cuniq, uint32_t *ccnt, EdgeRun *run);
// sorted canonical keys (duplicates and loops in) -> unique simple edges (+ optional multiplicities)
int unique_edges(kombgpu_ctx *ctx, const uint64_t *keys, uint64_t count, DevBuf<uint64_t> &edges, uint64_t *n_edges,
                 DevBuf<uint32_t> *mult);
// keys sorted by high word in [base, base + n_rows): start[x] = first index whose high word is >= base + x, x in [0, n_rows];
// long runs of empty rows are filled by whole CTAs.  *err_dev (optional) is set to 2 when a key is out of range or its
// low word is >= lo_bound.
int row_starts(kombgpu_ctx *ctx, const uint64_t *keys, uint64_t count, uint32_t base, uint32_t n_rows, uint32_t lo_bound, uint32_t *start,
               uint32_t *err_dev);
// fwd_start[x] = first edge whose source is >= x, x in [0, n]  (the edge list is sorted by source)
int forward_index(kombgpu_ctx *ctx, const uint64_t *edges, uint64_t n_edges, uint32_t n, uint32_t **fwd_start_out);
int swapped_sorted(kombgpu_ctx *ctx, const uint64_t *edges, uint64_t n_edges, uint32_t n_vertices, DevBuf<uint64_t> &a,
                   DevBuf<uint64_t> &b, uint64_t **out);
int lower_bounds_hi(kombgpu_ctx *ctx, const uint64_t *keys, uint64_t count, const uint32_t *bounds_host, int nb,
                    uint64_t *idx_host);
int csr_from_directed(kombgpu_ctx *ctx, const uint64_t *entries, uint64_t count, uint32_t v_lo, uint32_t n_local,
                      uint32_t n_global, uint64_t **row_ptr_out, uint32_t **col_out, int32_t **deg_out, int32_t *max_deg_out,
                      uint64_t *n_directed_out);

int csr_from_edges(kombgpu_ctx *ctx, DevBuf<uint64_t> &edges, uint64_t n_edges, uint32_t n, kombgpu_graph *g);

int adopt_csr(kombgpu_ctx *ctx, const uint64_t *row_ptr, const uint32_t *col, uint32_t n, kombgpu_graph *g);

// stage 2 (peel.cu)
int peel_coreness(kombgpu_graph *g);

// stage 3 (corea.cu) — device pointers in, device score out; *max_score on host
int corea_scores(kombgpu_ctx *ctx, const int32_t *core, const int32_t *deg, uint32_t n, int key_mode, double *score,
                 double *max_score_host);

// the maximal core and its truss (truss.cu), in three steps the partitioned graph (pcore.cu) runs apart:
// 1. sub_id[v] = compact id of v (~0 outside), core_vid = the original ids, for the n ids whose coreness is kmax
int max_core_vertices(kombgpu_ctx *ctx, const int32_t *core, uint32_t n, int32_t kmax, DevBuf<uint32_t> &sub_id,
                      DevBuf<uint32_t> &core_vid, uint32_t *n_core);
// 2. the edges of a canonical list (or of a slice of it) with both ends in the core, relabelled; the relabelling is
//    monotone, so the result stays canonical and sorted
int max_core_edges(kombgpu_ctx *ctx, const uint64_t *edges, uint64_t count, const uint32_t *sub_id, DevBuf<uint64_t> &out,
                   uint64_t *m);
// 3. the trussness of every edge of the canonical sub-edge list (m < 2^32) and the unitigs on the edges of maximal
//    trussness; on success sub_edges and core_vid move into *tr
int sub_edges_truss(kombgpu_ctx *ctx, DevBuf<uint64_t> &sub_edges, uint64_t m, DevBuf<uint32_t> &core_vid, uint32_t n_core,
                    MaxCoreTruss *tr);
// the cached result to the host (u, v: original ids; any pointer may be NULL)
int truss_edges_to_host(kombgpu_ctx *ctx, const MaxCoreTruss &tr, uint32_t *u, uint32_t *v, int32_t *trussness);
int truss_vertices_to_host(kombgpu_ctx *ctx, const MaxCoreTruss &tr, uint32_t *vids);
void truss_free(kombgpu_ctx *ctx, MaxCoreTruss *tr);

// densest k-core (densest.cu): hist[core[v]] += 1 over `count` vertices (edges == NULL), or hist[min(core[u], core[v])]
// += 1 over `count` edges of a canonical list; the k-core of the summed histograms with the largest density
int level_histogram(kombgpu_ctx *ctx, const int32_t *core, const uint64_t *edges, uint64_t count, uint32_t n_bins,
                    unsigned long long *hist);
struct DensestCore {
    int32_t k;
    uint64_t n_vertices, n_edges;
    double density;
};
// hv / he: histograms of n_bins levels over the n vertices and n_edges edges (unread when either count is 0)
DensestCore densest_level(const unsigned long long *hv, const unsigned long long *he, uint32_t n_bins, uint64_t n, uint64_t n_edges);

// densest block (densest.cu): the bulk greedy peel, shared by the single-GPU graph and the partitioned one (pcore.cu).
// pass[v] = the pass that removed v, kBlockUnset while v survives.
constexpr int kBlockThreads = 256;
constexpr uint32_t kBlockUnset = 0xffffffffu;
struct BlockPass {
    unsigned long long removed, single, both;   // unitigs removed; entries towards survivors / towards unitigs removed in the same pass
    double w_removed;
};
// over the n unitigs of a slice: pass[i] = t for every survivor with w[i] + deg_s[i] <= thr (w NULL: weights 0); their ids
// id_base + i go to list[st->removed ...], st->removed and st->w_removed count them
__global__ void __launch_bounds__(kBlockThreads) block_mark_kernel(const double *__restrict__ w, const int32_t *__restrict__ deg_s, uint32_t n,
                                                                   double thr, uint32_t t, uint32_t id_base, uint32_t *__restrict__ pass,
                                                                   uint32_t *__restrict__ list, BlockPass *__restrict__ st);
__global__ void __launch_bounds__(kBlockThreads) block_member_kernel(const uint32_t *__restrict__ pass, uint32_t n, uint32_t t_best,
                                                                     uint8_t *__restrict__ member);
inline uint32_t block_grid(const kombgpu_ctx *ctx, uint64_t n) {
    const uint32_t g = ceil_div_u64(n ? n : 1, kBlockThreads), cap = (uint32_t)ctx->sm_count * 8u;
    return g < cap ? g : cap;
}
// the sum of n weights on the device, by the mark kernel's reduction over a scratch pass map (list: n entries of room)
int block_weight_sum(kombgpu_ctx *ctx, const double *w, const int32_t *deg_s, uint32_t n, uint32_t *list, BlockPass *st, double *sum);
// pass[0, n) >= t_best to the host (n bytes)
int block_member(kombgpu_ctx *ctx, const uint32_t *pass, uint32_t n, uint32_t t_best, uint8_t *member);

// The two steps of one pass over the whole graph; densest_block_passes drives them.
struct BlockSteps {
    // pass t: remove every survivor with w(v) + deg_S(v) <= thr; h->removed and h->w_removed over the whole graph
    virtual int mark(double thr, uint32_t t, BlockPass *h) = 0;
    // the survivors lose their neighbours removed in pass t; h->single and h->both over the whole graph
    virtual int update(uint32_t t, BlockPass *h) = 0;
};
struct DensestBlock {
    uint64_t n_vertices, n_edges;
    double weight_sum, density;
    uint32_t passes, t_best;   // the block is {v : pass[v] >= t_best}
};
// the pass loop over a graph of n unitigs, n_edges edges and weight sum W: density and best block, threshold, the retry of
// an empty pass, the clamp of W and the pass limit
int densest_block_passes(kombgpu_ctx *ctx, uint64_t n, uint64_t n_edges, double W, double eps, BlockSteps &steps, DensestBlock *out);

#ifdef __CUDACC__
// one warp per removed unitig list[k]: it walks the unitig's neighbours nb[ptr[x] .. ptr[x + 1]) (ids into pass and deg_s).
// A survivor loses a neighbour; st->single counts the entries towards survivors, st->both those towards unitigs removed
// in the same pass t.
template <typename Ptr>
__device__ __forceinline__ void block_update_warps(const Ptr *__restrict__ ptr, const uint32_t *__restrict__ nb, const uint32_t *__restrict__ list,
                                                   uint32_t n_list, uint32_t t, const uint32_t *__restrict__ pass, int32_t *__restrict__ deg_s,
                                                   BlockPass *__restrict__ st) {
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5, lane = lane_id();
    unsigned long long single = 0, both = 0;
    for (uint32_t k = warp; k < n_list; k += n_warps) {
        const uint32_t i = list[k];
        const uint64_t lo = ptr[i], hi = ptr[i + 1];
        for (uint64_t e = lo + lane; e < hi; e += 32) {
            const uint32_t j = nb[e];
            const uint32_t pj = pass[j];
            if (pj == kBlockUnset) { atomicSub(&deg_s[j], 1); ++single; }
            else if (pj == t) ++both;
        }
    }
    single = warp_reduce_add(single);
    both = warp_reduce_add(both);
    if (lane == 0) {
        if (single) atomicAdd(&st->single, single);
        if (both) atomicAdd(&st->both, both);
    }
}
#endif

void graph_release(kombgpu_graph *g);
void truss_release(kombgpu_graph *g);   // truss.cu
void format_release(kombgpu_graph *g);  // format.cu

}  // namespace kg
