// dgraph.cuh — one rank's share of a unitig graph partitioned by unitig-id range over the ranks of a communicator
// (SURVEY.md section 8(e)); stage entry points of the partitioned path (pbuild.cu, ppeel.cu, pcorea.cu, format.cu).
#pragma once

#include "comm.cuh"
#include "graph.cuh"

// Sizes and device timings of one rank's share (kombgpu_dist_graph_stats)
struct kombgpu_dist_graph {
    kombgpu_comm *comm = nullptr;
    kombgpu_ctx *ctx = nullptr;
    uint32_t n_global = 0;
    uint32_t step = 1;         // rank q owns unitig ids [q * step, min((q + 1) * step, n_global))
    uint32_t v_lo = 0, n_local = 0;
    uint64_t n_fwd = 0;        // edges (u, v), u < v, whose u this rank owns: its slice of the canonical edge list
    uint64_t n_directed = 0;   // CSR entries of the local rows
    uint64_t n_edges_global = 0;
    uint32_t build_rounds = 0;     // rounds the build emitted, routed and reduced the pairs in (1: one shot)
    uint64_t *edges = nullptr;     // [n_fwd]  (u << 32 | v), global ids, ascending
    uint32_t *mult = nullptr;      // [n_fwd]
    uint32_t *fwd_start = nullptr; // [n_local + 1]
    // the local entries of the symmetric adjacency, grouped by NEIGHBOUR: for every unitig x of the whole graph,
    // nbr[nbr_ptr[x] .. nbr_ptr[x + 1]) are the LOCAL ids (u - v_lo) of the unitigs this rank owns that are adjacent to x.
    // (By symmetry this is the transpose of the rank's rows: when x is peeled, these are the degrees this rank decrements.)
    uint32_t *nbr_ptr = nullptr;   // [n_global + 1]
    uint32_t *nbr = nullptr;       // [n_directed]
    // ... or, for the asynchronous peel (apeel.cu), as the rank's ROWS: col[row_ptr32[u] .. row_ptr32[u + 1]) are the global
    // ids of the neighbours of local unitig u (rows need no order inside).  A build makes one of the two layouts.
    uint32_t *row_ptr32 = nullptr; // [n_local + 1]
    uint32_t *col = nullptr;       // [n_directed]
    int peel_choice = 0;           // what the build prepared for: 0 log-based (ppeel.cu), 1 asynchronous (apeel.cu), 2 replicated (rpeel.cu)
    int32_t *deg = nullptr;        // [n_local]
    int32_t *core = nullptr;       // [n_local] after the peel
    double *score = nullptr;       // [n_local] after CORE-A
    bool has_core = false, has_score = false;
    double max_score = 0.0;        // global
    // the maximal core of the WHOLE graph and the trussness of its edges, the same on every rank (pcore.cu)
    bool has_truss = false;
    kg::MaxCoreTruss tr;
    float ms_truss[3] = {0.f, 0.f, 0.f};   // CUDA-event times: coreness gather, selection + slice gather, truss peel
    // this rank's slices of the three output files, formatted on the device (format.cu), cached until destroy
    char *text[3] = {nullptr, nullptr, nullptr};
    uint64_t text_bytes[3] = {0, 0, 0};
    kombgpu_dist_stats st{};
};

namespace kg {

inline uint32_t owner_step(uint32_t n_global, int world) { return n_global ? (n_global + (uint32_t)world - 1) / (uint32_t)world : 1u; }

// pbuild.cu: local hits / pairs -> this rank's rows
int dist_build(kombgpu_comm *c, const uint32_t *a, const uint32_t *b, uint64_t count, uint32_t n_global, bool from_hits,
               kombgpu_dist_graph *g);
// send every key to the rank that owns its high word (hi / step); returns the keys this rank received, in the
// symmetric heap (valid until the caller's sym_release).  kRebase: the high word arrives as hi - owner * step.
// local_rc: this rank has already failed with that code; it sends nothing, and every rank returns an error (the
// failing rank its own code and message, the others the code of the first failing rank).
int route_keys(kombgpu_comm *c, const uint64_t *keys, uint64_t n, uint32_t step, bool rebase, uint64_t **recv, uint64_t *n_recv,
               int local_rc = KOMBGPU_OK);
// ppeel.cu
int dist_peel(kombgpu_dist_graph *g);
// apeel.cu
int dist_peel_async(kombgpu_dist_graph *g);
// rpeel.cu
int dist_peel_replicated(kombgpu_dist_graph *g);
// which peel a build prepares for (pbuild.cu): KOMBGPU_DIST_PEEL = log (ranks meet once per cascade generation, ppeel.cu),
// async (apeel.cu), replicated (rpeel.cu) or auto (default: by the shape of the graph).  0 log, 1 async, 2 auto, 3 replicated.
int dist_peel_mode();
// pcorea.cu
int dist_corea(kombgpu_dist_graph *g, int key_mode);
// pcore.cu: the consumers of the finished coreness
int dist_max_core_truss(kombgpu_dist_graph *g);
int dist_densest_core(kombgpu_dist_graph *g, DensestCore *out);
// weight: this rank's slice (host, or NULL); member: this rank's slice (host, n_local bytes, or NULL)
int dist_densest_block(kombgpu_dist_graph *g, const double *weight, int use_scores, double eps, DensestBlock *out, uint8_t *member);

// psam.cu: the names of the vertices [v_lo, v_lo + n_local) a kombgpu_dist_hits holds on this rank's device:
// name i is bytes[off[i] .. off[i] + len[i])
struct DistNames {
    const kombgpu_comm *comm;
    uint32_t n_unitigs, v_lo, n_local;
    const unsigned char *bytes;
    const uint64_t *off;
    const uint32_t *len;
};
int dist_hits_name_text(const kombgpu_dist_hits *h, DistNames *out);
// format.cu
void dist_format_release(kombgpu_dist_graph *g);

void dist_graph_release(kombgpu_dist_graph *g);

}  // namespace kg
