/*
 * kombgpu.h — C ABI of the B200-native KOMB hot path
 *             (hits -> unitig adjacency graph -> k-core -> CORE-A).
 *
 * The reference (treangenlab/komb, komb2) has no FFI: its hot path is reached
 * through the C++ methods of komb::Kgraph (src/graph.h:49-62) called in a fixed
 * order from main (src/komb2.cpp:93-132).  This header is the boundary a
 * maintainer binds instead (see INTEGRATION.md): it starts where the reference
 * holds tokenised hits (after src/graph.cpp:221-235) and ends where it formats
 * its three output files (src/graph.cpp:423-426,467-475; CombineCoreA.h:36-39).
 *
 * Conventions
 *   - every function returns 0 (KOMBGPU_OK) or a negative KOMBGPU_E* code;
 *     nothing throws or exits across the ABI; kombgpu_last_error() gives text.
 *   - plain pointers + sizes only.  Pointers are HOST pointers unless the
 *     function name ends in `_dev` (then they are device pointers on the
 *     context's device, e.g. a torch tensor's data_ptr()).
 *   - the caller owns every buffer it passes; the library owns device memory
 *     behind the opaque handles.  One context per process and device; calls on
 *     one context are serialised by the caller.
 *   - there is NO CPU fallback: without a usable CUDA device every compute
 *     entry point fails with KOMBGPU_ENODEV.
 */
#ifndef KOMBGPU_H
#define KOMBGPU_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KOMBGPU_ABI_VERSION 1

enum {
    KOMBGPU_OK = 0,
    KOMBGPU_EINVAL = -1,  /* bad argument (null pointer, id out of range, ...)   */
    KOMBGPU_ENODEV = -2,  /* no usable CUDA device / device is not sm_100        */
    KOMBGPU_ENOMEM = -3,  /* device or host allocation failed                    */
    KOMBGPU_ECUDA = -4,   /* a CUDA call or kernel failed (see last_error)       */
    KOMBGPU_ESTATE = -5,  /* call order violated (e.g. corea before coreness)    */
    KOMBGPU_EINTERNAL = -6 /* internal invariant broken (peel watchdog tripped)  */
};

/* CORE-A key arithmetic (SURVEY.md quirk Q5, reference src/CoreA.h:122).  Both modes take any coreness and degree
 * in [0, 2^31), degrees >= n included: exact64 ranks the int64 value coreness * n + degree, so a degree >= n carries
 * into the coreness exactly as in that sum (with n = 4, (coreness 0, degree 5) ranks above (1, 0)). */
enum {
    KOMBGPU_KEY_REF32 = 0,   /* (int32)(coreness * n + degree), wraps like the reference */
    KOMBGPU_KEY_EXACT64 = 1  /* the same expression in int64, without overflow            */
};

typedef struct kombgpu_ctx kombgpu_ctx;
typedef struct kombgpu_graph kombgpu_graph;

/* Sizes and device timings of the last operations on a graph. */
typedef struct kombgpu_stats {
    uint64_t n_hits;         /* H: hits passed to build_graph                          */
    uint64_t n_unique_hits;  /* distinct (read, unitig)                                */
    uint64_t n_pairs;        /* P: clique pairs emitted before dedup (or m for from_edges) */
    uint64_t n_edges;        /* E: simple undirected edges                             */
    uint32_t n_vertices;     /* n                                                      */
    int32_t max_degree;
    int32_t max_coreness;    /* -1 until kombgpu_coreness ran                          */
    uint32_t peel_levels;    /* non-empty coreness levels processed                    */
    uint32_t peel_rounds;    /* grid-wide dependent rounds (scan+process phases)       */
    float ms_build;          /* CUDA-event time: hits/edges -> CSR                     */
    float ms_peel;           /* CUDA-event time: k-core peel                           */
    float ms_corea;          /* CUDA-event time: CORE-A                                */
    float ms_peel_kernel;    /* CUDA-event time of the persistent peel kernel alone    */
    uint64_t kernel_launches; /* kernels of this library launched for this graph       */
} kombgpu_stats;

/* ---- context ------------------------------------------------------------- */

/* Create a context on CUDA device `device` (a CUDA ordinal).  Replaces the
 * reference's `komb::Kgraph(threads, readlen)` constructor (src/graph.cpp:52-56,
 * src/komb2.cpp:79) as the per-process state holder. */
int kombgpu_ctx_create(int device, kombgpu_ctx **out);
void kombgpu_ctx_destroy(kombgpu_ctx *ctx);

/* Run all work of this context on an existing CUDA stream (a cudaStream_t cast
 * to void*, e.g. torch.cuda.current_stream().cuda_stream).  As everywhere in
 * CUDA, NULL is the legacy default stream (which is what torch uses unless told
 * otherwise).  kombgpu_ctx_reset_stream returns to the context's private
 * non-blocking stream (the state after kombgpu_ctx_create). */
int kombgpu_ctx_set_stream(kombgpu_ctx *ctx, void *cuda_stream);
int kombgpu_ctx_reset_stream(kombgpu_ctx *ctx);

/* Text of the last error on this context (never NULL).  With ctx == NULL:
 * the last error of a failed kombgpu_ctx_create on this thread. */
const char *kombgpu_last_error(const kombgpu_ctx *ctx);

/* Page-locked host memory for the buffers a host passes to the copying entry
 * points (hits in, edges / degree / coreness / score out): DMA at full PCIe rate
 * instead of staged pageable copies.  A host without CUDA headers can use these. */
int kombgpu_pinned_alloc(kombgpu_ctx *ctx, uint64_t bytes, void **out);
int kombgpu_pinned_free(kombgpu_ctx *ctx, void *ptr);

/* Number of this library's kernels launched through the context so far. */
int kombgpu_ctx_launches(const kombgpu_ctx *ctx, uint64_t *launches);

/* Release cached device workspace held by the context. */
int kombgpu_ctx_trim(kombgpu_ctx *ctx);

/* ---- stage 1: graph build ------------------------------------------------- */

/* Hits of BOTH mate files, concatenated: hit i = read `read_key[i]` aligned to
 * unitig `unitig[i]` (< n_vertices).  Builds the simple undirected unitig graph:
 * per-read union of unitig sets, every set a clique, duplicates and loops
 * dropped.  Replaces Kgraph::getEdgeInfo + generateGraph + igraph_create +
 * igraph_simplify (src/graph.cpp:259-285, 287-393, 418, 438).
 * Limits on one device: n_hits < 2^32, distinct (read, unitig) hits < 2^31 and simple edges < 2^32
 * (KOMBGPU_EINVAL otherwise).  The clique pairs P (kombgpu_stats.n_pairs, C(k, 2) for a read with k unitigs)
 * are not limited: from P >= 2^32 on they are emitted, sorted and reduced in chunks of fewer than 2^30 pairs and
 * merged into the edge list, so device memory stays at one chunk plus O(edges + hits).  The results do not
 * depend on the chunking. */
int kombgpu_build_graph(kombgpu_ctx *ctx, const uint32_t *read_key, const uint32_t *unitig,
                        uint64_t n_hits, uint32_t n_vertices, kombgpu_graph **out);
int kombgpu_build_graph_dev(kombgpu_ctx *ctx, const uint32_t *read_key_dev, const uint32_t *unitig_dev,
                            uint64_t n_hits, uint32_t n_vertices, kombgpu_graph **out);

/* Arbitrary (u, v) pairs, ids < n_vertices; duplicates, both orientations and
 * self-loops allowed.  Replaces igraph_create + igraph_simplify
 * (src/graph.cpp:418, 438) for an edge list that already exists.
 * n_pairs is not limited (pairs from 2^32 on are reduced in chunks, as in kombgpu_build_graph); simple edges
 * must stay below 2^32.  An edge's multiplicity (kombgpu_graph_edge_multiplicity) saturates at 2^32 - 1 when
 * it occurs that often or more.  The host-pointer variant uploads the whole input first. */
int kombgpu_graph_from_edges(kombgpu_ctx *ctx, const uint32_t *u, const uint32_t *v,
                             uint64_t n_pairs, uint32_t n_vertices, kombgpu_graph **out);
int kombgpu_graph_from_edges_dev(kombgpu_ctx *ctx, const uint32_t *u_dev, const uint32_t *v_dev,
                                 uint64_t n_pairs, uint32_t n_vertices, kombgpu_graph **out);

/* Adopt an existing CSR of a simple symmetric graph (device pointers; row_ptr[n+1],
 * col[row_ptr[n]], rows need not be sorted).  The arrays are copied.  Used by the
 * multi-GPU path after all-gathering the rank-local rows; the canonical edge
 * list is not materialised (kombgpu_graph_edges returns KOMBGPU_ESTATE). */
int kombgpu_graph_from_csr_dev(kombgpu_ctx *ctx, const uint64_t *row_ptr_dev, const uint32_t *col_dev,
                               uint32_t n_vertices, kombgpu_graph **out);

void kombgpu_graph_destroy(kombgpu_graph *g);

/* |V| and |E| of the simple graph (igraph_vcount / igraph_ecount,
 * src/graph.cpp:443-444). */
int kombgpu_graph_counts(const kombgpu_graph *g, uint32_t *n_vertices, uint64_t *n_edges);

/* Canonical edge list: u[i] < v[i], ascending by (u, v); each array holds
 * n_edges entries.  This is what the drop-in writes to edgelist.txt (quirk Q7). */
int kombgpu_graph_edges(const kombgpu_graph *g, uint32_t *u, uint32_t *v);

/* The same edge list in CSR form, half the bytes: edge i is (u, v[i]) for the u with
 * fwd_ptr[u] <= i < fwd_ptr[u + 1]; fwd_ptr holds n_vertices + 1 entries, v holds n_edges. */
int kombgpu_graph_edges_csr(const kombgpu_graph *g, uint64_t *fwd_ptr, uint32_t *v);

/* Edge multiplicities, aligned with the canonical edge list: mult[i] = number of clique pairs (reads
 * holding both unitigs; or duplicate input pairs for kombgpu_graph_from_edges) that collapsed into edge i.
 * An extension: the reference drops duplicates without counting them (igraph_simplify with comb = NULL,
 * src/graph.cpp:438); the sum over all edges equals kombgpu_stats.n_pairs minus the self-loops. */
int kombgpu_graph_edge_multiplicity(const kombgpu_graph *g, uint32_t *mult);

/* CSR of the symmetric graph: row_ptr[n+1], col[2E], every row ascending. */
int kombgpu_graph_csr(const kombgpu_graph *g, uint64_t *row_ptr, uint32_t *col);

/* ---- SAM text -> hits on the device (SURVEY.md section 8, row N1) ------------------------------------------
 *
 * The tokenising half of Kgraph::readSAM (src/graph.cpp:197-239, at -t 1: '@' lines skipped, tokens 0 and 2 under
 * strtok("\t") rules, RNAME "*" skipped, read key = QNAME.substr(1, QNAME.find('/')), an unterminated final line
 * is not processed) and the merge + vid assignment that follows it (src/graph.cpp:242-256), for a host that
 * hands over the raw bytes of its SAM files instead of tokenising them itself.  `texts[f]` / `sizes[f]` are the
 * bytes of input f (host pointers; mate 1 first).  Numbering is deterministic, unlike the reference's (quirk Q4):
 * read ids follow first appearance; unitig ids follow @SQ header order, then first appearance, over unitigs with
 * at least one hit.  Strings are matched by their bytes, never by hash alone.  Empty lines and lines with fewer
 * than three tokens (undefined behaviour in the reference) fail with KOMBGPU_EINVAL; so do more than 2^30 lines in
 * one call.  The hits stay on the
 * device: kombgpu_build_graph_hits builds the graph from them without a host round trip. */
typedef struct kombgpu_hits kombgpu_hits;
int kombgpu_sam_parse(kombgpu_ctx *ctx, const char *const *texts, const uint64_t *sizes, int n_files, kombgpu_hits **out);
void kombgpu_hits_destroy(kombgpu_hits *hits);
/* hits, distinct read keys, unitigs with a hit (= vertices), terminated lines seen; any pointer may be NULL */
int kombgpu_hits_counts(const kombgpu_hits *hits, uint64_t *n_hits, uint32_t *n_reads, uint32_t *n_unitigs, uint64_t *n_lines);
/* Name of every vertex as a span of the inputs: bytes [offset[v], offset[v] + len[v]) of input file[v]
 * (n_unitigs entries each; `file` may be NULL).  The host keeps the strings, the device keeps the ids. */
int kombgpu_hits_names(const kombgpu_hits *hits, uint32_t *file, uint64_t *offset, uint32_t *len);
/* The integer hits in file order (n_hits entries each; either pointer may be NULL). */
int kombgpu_hits_download(const kombgpu_hits *hits, uint32_t *read_key, uint32_t *unitig);
int kombgpu_hits_device_arrays(const kombgpu_hits *hits, const uint32_t **read_key_dev, const uint32_t **unitig_dev);
/* CUDA-event times of the upload and of the parse + interning kernels, kernels launched, hash seeds tried */
int kombgpu_hits_timing(const kombgpu_hits *hits, float *ms_upload, float *ms_parse, uint64_t *kernel_launches, int *hash_rounds);
/* kombgpu_build_graph_dev on the device-resident hits */
int kombgpu_build_graph_hits(const kombgpu_hits *hits, kombgpu_graph **out);

/* ---- stage 2: degree + coreness ------------------------------------------- */

/* igraph_degree(ALL, NO_LOOPS) (src/graph.cpp:462): degree[n]. */
int kombgpu_degree(const kombgpu_graph *g, int32_t *degree);

/* igraph_coreness(ALL) (src/graph.cpp:463): runs the frontier peel on first
 * call, then copies coreness[n] to the host (coreness may be NULL to only run). */
int kombgpu_coreness(kombgpu_graph *g, int32_t *coreness);

/* ---- stage 3: CORE-A ------------------------------------------------------- */

/* CoreA::getAnomalyScore (src/CoreA.h:109-140) on host arrays:
 * score[i] = |ln rank(degree)[i] - ln rank(key)[i]|, descending average-tie
 * ranks (src/CoreA.h:142-187). */
int kombgpu_corea(kombgpu_ctx *ctx, const int32_t *coreness, const int32_t *degree,
                  uint32_t n, int key_mode, double *score);

/* The same on the device-resident coreness/degree of a graph (requires
 * kombgpu_coreness first).  score may be NULL to only run. */
int kombgpu_graph_corea(kombgpu_graph *g, int key_mode, double *score);

/* The two scalars CombineCoreA::run prints (src/CombineCoreA.h:24-25,31-32):
 * max coreness (dense ratio = max_coreness / 2, integer division) and the max
 * CORE-A score. */
int kombgpu_graph_summary(const kombgpu_graph *g, int32_t *max_coreness, double *max_score);

/* ---- output files formatted on the device (SURVEY.md section 8, row N2) ----------------------------------
 *
 * The bytes of the three files the reference writes with one fprintf per row: edgelist.txt "%d\t%d\n" per simple
 * edge in canonical order (src/graph.cpp:423-426; quirk Q7), kcore.tsv "#VID\tName\tCoreness\tDegree\n" +
 * "%d\t%s\t%d\t%d\n" per unitig (src/graph.cpp:467-475) and CoreA_anomaly.txt "%d\t%f\n" per unitig
 * (src/CombineCoreA.h:36-39; "%f" as glibc prints it: six decimals of the exact binary value, ties to even).
 * kombgpu_graph_format formats file `which` on the device and reports its size; kombgpu_graph_format_fetch copies
 * it to the host -- with async != 0 on the copy stream, so that compute issued afterwards (the peel under the
 * edge-list download) overlaps it; kombgpu_graph_format_wait ends the asynchronous copies.  KCORE needs the
 * coreness and the kombgpu_hits the graph was built from (the names live in its copy of the SAM text); COREA
 * needs the scores.  The host issues one write per file. */
enum { KOMBGPU_FILE_EDGELIST = 0, KOMBGPU_FILE_KCORE = 1, KOMBGPU_FILE_COREA = 2 };
int kombgpu_graph_format(kombgpu_graph *g, int which, const kombgpu_hits *names, uint64_t *bytes);
int kombgpu_graph_format_fetch(kombgpu_graph *g, int which, char *dst, int async);
int kombgpu_graph_format_wait(kombgpu_graph *g);
/* CoreA_anomaly.txt from a host array of scores (finite, |score| < 2^43): *bytes = size of the text; it is
 * copied to dst when it fits `capacity` (else KOMBGPU_EINVAL, *bytes still set). */
int kombgpu_format_corea(kombgpu_ctx *ctx, const double *score, uint32_t n, char *dst, uint64_t capacity, uint64_t *bytes);

/* ---- whole path + introspection --------------------------------------------- */

/* build (already done) -> coreness -> CORE-A in one call, results left on the
 * device; the three getters above then only copy. */
int kombgpu_graph_analyse(kombgpu_graph *g, int key_mode);

/* Everything the komb2 host writes to its three files, in one call: runs the peel and
 * CORE-A if they have not run yet and copies the canonical edge list (u, v: n_edges
 * entries each), degree, coreness and score (n_vertices entries each) to the host.
 * The edge list (most of the bytes) is downloaded on a copy stream WHILE the peel
 * runs; with page-locked buffers (kombgpu_pinned_alloc) that copy is free.
 * Any output pointer may be NULL (u and v only together). */
int kombgpu_graph_results(kombgpu_graph *g, int key_mode, uint32_t *u, uint32_t *v, int32_t *degree,
                          int32_t *coreness, double *score);

/* kombgpu_graph_results with the edge list in CSR form (see kombgpu_graph_edges_csr): n_vertices + 1
 * offsets and n_edges targets instead of two arrays of n_edges -- half the device-to-host bytes. */
int kombgpu_graph_results_csr(kombgpu_graph *g, int key_mode, uint64_t *fwd_ptr, uint32_t *v, int32_t *degree,
                              int32_t *coreness, double *score);

/* Densest k-core (needs kombgpu_coreness): the level k* whose core {v : coreness(v) >= k*} maximises
 * edges / vertices, with that block's size.  Bulk analogue of the greedy densest-block peel the reference keeps,
 * unreachable from main, in CombineCoreA::runMerge over HashIndexedMinHeap (src/CombineCoreA.h:45-219,
 * src/HashIndexedMinHeap.h:10-238) for suspiciousness == nullptr: same density (2E directed entries over 2V row
 * and column nodes), blocks restricted to the nested k-cores (still a 2-approximation of the densest subgraph),
 * ties to the largest block.  The reference's own result depends on heap tie order and uninitialised memory, so
 * there is no parity obligation (SURVEY.md section 8, row A9). */
int kombgpu_graph_densest_core(kombgpu_graph *g, int32_t *k_star, uint32_t *n_vertices, uint64_t *n_edges,
                               double *density);

/* Densest BLOCK: the greedy peel of CombineCoreA::runMerge (src/CombineCoreA.h:45-219, over HashIndexedMinHeap,
 * src/HashIndexedMinHeap.h:10-238) in bulk form.  f(S) = sum of the unitigs' weights + edges inside S, density =
 * f(S) / |S| (the reference's suspiciousSum / nodes left: both counted twice there, once per row / column copy),
 * priority(v) = weight(v) + degree inside S.  The reference removes the minimum-priority node one at a time; here a
 * pass removes every survivor with priority <= 2 (1 + eps) density(S) (at least an eps / (1 + eps) share of them),
 * and the densest S seen is returned: a 2 (1 + eps)-approximation of the densest block (2 for the serial order), in
 * O(log n / eps) passes, independent of any tie order.  `weight`: n_vertices host doubles >= 0 (the reference's
 * `suspiciousness`), or NULL with use_scores != 0 for the graph's own CORE-A scores, or NULL / 0 for the unweighted
 * peel.  member (optional): n_vertices bytes, 1 for the unitigs of the block.  Any output pointer may be NULL. */
int kombgpu_graph_densest_block(kombgpu_graph *g, const double *weight, int use_scores, double eps, uint32_t *n_vertices,
                                uint64_t *n_edges, double *weight_sum, double *density, uint32_t *n_passes, uint8_t *member);

/* The maximal core and the trussness of its edges (needs kombgpu_coreness): the induced subgraph of the unitigs
 * whose coreness is the maximum, igraph_trussness of every edge of it (the largest k such that the edge lies in a
 * k-truss; 2 for an edge in no triangle) and the unitigs on the edges of maximal trussness -- what the reference's
 * Kgraph::runTruss computes before it writes truss_unitigs.fasta (src/graph.cpp:486-563; runCore collects the
 * maximal core at :470-476; the call is commented out at :478).  Computed once per graph, cached. */
int kombgpu_graph_max_core_truss(kombgpu_graph *g, uint32_t *n_core_vertices, uint64_t *n_core_edges,
                                 int32_t *max_trussness, uint32_t *n_truss_vertices);
/* Edges of the maximal core (original unitig ids, u < v, ascending) with their trussness; n_core_edges entries each. */
int kombgpu_graph_max_core_edges(const kombgpu_graph *g, uint32_t *u, uint32_t *v, int32_t *trussness);
/* The unitigs on edges of maximal trussness (original ids, ascending); n_truss_vertices entries. */
int kombgpu_graph_truss_vertices(const kombgpu_graph *g, uint32_t *vids);

/* ---- the unitig FASTA: sequences of the unitigs the analysis singles out --------------------------------------
 *
 * FASTA records.  The input is the bytes of one FASTA file.  A record starts at a '>' at offset 0 or right after a
 * '\n' and ends where the next record starts, or at the end of the file.  Its name is the bytes after '>' up to the
 * first of ' ' '\t' '\r' '\n' '\v' '\f' -- the rule by which bwa-mem2 (kseq) derives the SAM RNAME, so names in the
 * FASTA match RNAMEs in the SAM.  Sequence lines are never parsed: wrapped records, CRLF line endings and header
 * descriptions pass through unchanged.  KOMBGPU_EINVAL, with a message, for non-whitespace bytes before the first
 * record, an empty name, or two records with the same name (the join would be ambiguous).  An empty file has zero
 * records.
 *
 * Join.  Every vertex gets the record whose name equals its unitig name, compared byte for byte (a hash alone never
 * decides a match).  Vertices without a record are counted (*n_missing); that is not an error at join time.
 *
 * Anomalous unitigs (IQR fence on CORE-A).  s = the n scores sorted ascending; each quartile as
 * numpy.percentile(..., method="linear") computes it, in float64: h = n p - p for p = 0.25 and 0.75, i = floor(h),
 * j = min(i + 1, n - 1), t = h - i, d = s[j] - s[i], q = s[i] + d t when t < 0.5, else q = s[j] - d (1 - t).  Then
 * fence = q3 + whisker (q3 - q1), and vertex v is anomalous iff score[v] > fence (strictly); whisker is usually 1.5.
 * NaN scores are KOMBGPU_EINVAL; negative scores are allowed; n = 0 selects nothing and reports zeros.  There is no
 * parity claim against the reference's getMedian / splitAnomalousUnitigs: their sources are not in this tree and the
 * reference disables them; the rule above is the spec.
 *
 * Extraction.  The bytes of the selected vertices' records, copied verbatim, in the order of the FASTA file; a '\n' is
 * appended only when the file's last record is unterminated and selected.  A selected vertex without a record is
 * KOMBGPU_EINVAL, and the message names one such vertex id and its unitig name.  The output stays on the device until
 * kombgpu_fasta_extract_fetch copies it (into page-locked memory from kombgpu_pinned_alloc for full PCIe rate). */
typedef struct kombgpu_fasta kombgpu_fasta;
/* Upload `size` bytes of FASTA text and index its records on the device. */
int kombgpu_fasta_load(kombgpu_ctx *ctx, const char *text, uint64_t size, kombgpu_fasta **out);
void kombgpu_fasta_destroy(kombgpu_fasta *fa);
/* records and bytes of the file; either pointer may be NULL */
int kombgpu_fasta_counts(const kombgpu_fasta *fa, uint32_t *n_records, uint64_t *n_bytes);
/* vertex -> record.  The vertex names are those of the kombgpu_hits the graph was built from (spans of its device copy
 * of the SAM text; same context), or a packed host table: name v is bytes [offsets[v], offsets[v + 1]) of `bytes`
 * (n + 1 offsets).  A join replaces the previous one. */
int kombgpu_fasta_join_hits(kombgpu_fasta *fa, const kombgpu_hits *names, uint32_t *n_missing);
int kombgpu_fasta_join_names(kombgpu_fasta *fa, const char *bytes, const uint64_t *offsets, uint32_t n, uint32_t *n_missing);
/* mask: n host bytes, nonzero = selected, n = the vertices of the last join; *bytes = size of the output text */
int kombgpu_fasta_extract(kombgpu_fasta *fa, const uint8_t *mask, uint32_t n, uint64_t *bytes);
int kombgpu_fasta_extract_fetch(kombgpu_fasta *fa, char *dst);
/* CUDA-event times of the upload, the index (record starts, names, table), the last join and the last extraction, and
 * the kernels launched for this FASTA; any pointer may be NULL */
int kombgpu_fasta_timing(const kombgpu_fasta *fa, float *ms_upload, float *ms_index, float *ms_join, float *ms_extract,
                         uint64_t *kernel_launches);
/* IQR fence on CORE-A over n host scores, or over the graph's own (needs kombgpu_graph_corea first, else
 * KOMBGPU_ESTATE).  member (optional): n bytes, 1 for the anomalous unitigs.  Any output pointer may be NULL. */
int kombgpu_anomalous(kombgpu_ctx *ctx, const double *score, uint32_t n, double whisker, double *q1, double *q3,
                      double *fence, uint32_t *n_selected, uint8_t *member);
int kombgpu_graph_anomalous(kombgpu_graph *g, double whisker, double *q1, double *q3, double *fence,
                            uint32_t *n_selected, uint8_t *member);

/* The whole path in one call, host buffers in and out: what komb2 does between readSAM and its three writers
 * (getEdgeInfo ... anomalyDetection, src/komb2.cpp:104-132).  Same results as kombgpu_build_graph followed by
 * kombgpu_graph_results; the difference is scheduling: the edge list is final half-way through the build (the CSR
 * only indexes it), so its download starts there and runs under the rest of the build, the peel and CORE-A.
 * u / v (both or neither) must hold edge_capacity entries; more edges than that is KOMBGPU_EINVAL (build with
 * kombgpu_build_graph and size the buffers from kombgpu_graph_counts instead).  Any output pointer may be NULL.
 * On success *out owns the device graph (kombgpu_graph_destroy). */
int kombgpu_analyse_hits(kombgpu_ctx *ctx, const uint32_t *read_key, const uint32_t *unitig, uint64_t n_hits,
                         uint32_t n_vertices, int key_mode, uint64_t edge_capacity, uint32_t *u, uint32_t *v,
                         int32_t *degree, int32_t *coreness, double *score, kombgpu_graph **out);

/* kombgpu_analyse_hits with the edge list in CSR form: fwd_ptr[n_vertices + 1], v[edge_capacity]. */
int kombgpu_analyse_hits_csr(kombgpu_ctx *ctx, const uint32_t *read_key, const uint32_t *unitig, uint64_t n_hits,
                             uint32_t n_vertices, int key_mode, uint64_t edge_capacity, uint64_t *fwd_ptr, uint32_t *v,
                             int32_t *degree, int32_t *coreness, double *score, kombgpu_graph **out);

int kombgpu_graph_stats(const kombgpu_graph *g, kombgpu_stats *out);

/* Device pointers of the graph's arrays (valid until kombgpu_graph_destroy);
 * any out-pointer may be NULL.  coreness/score are NULL until computed. */
int kombgpu_graph_device_arrays(const kombgpu_graph *g, const uint64_t **row_ptr, const uint32_t **col,
                                const uint64_t **edges_packed, const int32_t **degree,
                                const int32_t **coreness, const double **score);

/* ---- multi-GPU: one rank's share of a graph partitioned by unitig-id range --------
 *
 * One process per GPU; the exchanges between the calls below are done by the host
 * (torch.distributed / NCCL in komb_b200/distributed.py, MPI or ncclSend/Recv in
 * a C++ host).  `bounds[0..n_parts]` are the vertex-range boundaries: rank j owns
 * unitig ids [bounds[j], bounds[j+1]).  All pointers in this section whose name
 * ends in _dev are device pointers; counts and scalars are host pointers.
 *
 *   stage 1  every rank: its reads' hits -> local simple edge set  (kombgpu_local_edges_dev)
 *            route both directions of every edge to the owner of the source
 *            (kombgpu_edgeset_route_dev) -> all-to-all -> kombgpu_part_build_dev
 *   stage 2  per level k: kombgpu_part_peel_scan; then sub-rounds of
 *            kombgpu_part_peel_process (local cascade, remote targets to the outbox)
 *            -> kombgpu_part_outbox_route_dev -> all-to-all -> kombgpu_part_peel_apply_dev
 *            until no rank has a frontier or an outbox entry left
 *   stage 3  all-gather (coreness, degree) -> kombgpu_corea_dev
 */
typedef struct kombgpu_edgeset kombgpu_edgeset;
typedef struct kombgpu_part kombgpu_part;

/* Hits of this rank's reads (global unitig ids) -> sorted unique simple edges, kept
 * on the device.  Same semantics as kombgpu_build_graph up to the edge list. */
int kombgpu_local_edges_dev(kombgpu_ctx *ctx, const uint32_t *read_key_dev, const uint32_t *unitig_dev,
                            uint64_t n_hits, uint32_t n_vertices_global, kombgpu_edgeset **out);
/* The same from arbitrary (u, v) pairs (R-MAT style inputs). */
int kombgpu_edgeset_from_pairs_dev(kombgpu_ctx *ctx, const uint32_t *u_dev, const uint32_t *v_dev, uint64_t n_pairs,
                                   uint32_t n_vertices_global, kombgpu_edgeset **out);
int kombgpu_edgeset_counts(const kombgpu_edgeset *es, uint64_t *n_edges, uint64_t *n_pairs, uint64_t *n_unique_hits);
/* Directed entries (src << 32 | dst), both directions of every local edge, grouped
 * by the owner of src.  send_dev holds 2 * n_edges entries; counts[n_parts]. */
int kombgpu_edgeset_route_dev(kombgpu_edgeset *es, const uint32_t *bounds, int n_parts, uint64_t *send_dev,
                              uint64_t *counts);
void kombgpu_edgeset_destroy(kombgpu_edgeset *es);

/* Received directed entries with src in [v_lo, v_hi) (duplicates allowed: the same
 * edge may have been seen by several ranks) -> this rank's CSR rows. */
int kombgpu_part_build_dev(kombgpu_ctx *ctx, const uint64_t *entries_dev, uint64_t count, uint32_t v_lo,
                           uint32_t v_hi, uint32_t n_vertices_global, kombgpu_part **out);
void kombgpu_part_destroy(kombgpu_part *part);
int kombgpu_part_counts(const kombgpu_part *part, uint32_t *n_local, uint64_t *n_directed, int32_t *max_degree);
/* row_ptr[n_local+1], col[n_directed] (global ids), degree[n_local], coreness[n_local]
 * (working degrees during the peel, the coreness once it ended). */
int kombgpu_part_device_arrays(const kombgpu_part *part, const uint64_t **row_ptr, const uint32_t **col,
                               const int32_t **degree, const int32_t **coreness);

int kombgpu_part_peel_begin(kombgpu_part *part);
/* Level k: compact the local alive list; n_front local vertices at degree k,
 * n_alive above it, min_next = smallest degree above k (INT32_MAX if none). */
int kombgpu_part_peel_scan(kombgpu_part *part, int32_t k, uint32_t *n_front, uint32_t *n_alive, int32_t *min_next);
/* Peel the local frontier of level k including its local cascade; decrements of
 * vertices other ranks own are collected in the outbox (*n_outbox entries). */
int kombgpu_part_peel_process(kombgpu_part *part, int32_t k, uint32_t *n_outbox);
/* Outbox grouped by owner: send_dev holds n_outbox global ids; counts[n_parts]. */
int kombgpu_part_outbox_route_dev(kombgpu_part *part, const uint32_t *bounds, int n_parts, uint32_t *send_dev,
                                  uint64_t *counts);
/* Apply received decrements (global ids of vertices this rank owns); vertices that
 * reach degree k form the new local frontier (*n_front). */
int kombgpu_part_peel_apply_dev(kombgpu_part *part, int32_t k, const uint32_t *recv_dev, uint64_t count,
                                uint32_t *n_front);

/* kombgpu_corea on device arrays (score_dev[n]); *max_score on the host. */
int kombgpu_corea_dev(kombgpu_ctx *ctx, const int32_t *coreness_dev, const int32_t *degree_dev, uint32_t n,
                      int key_mode, double *score_dev, double *max_score);


/* ---- multi-GPU, peer-memory path: the whole hot path over the GPUs of one node -------------------------------
 *
 * One rank per GPU (one process per rank, or one host thread per rank inside one process).  The graph is
 * partitioned by unitig-id range: rank q owns ids [q * step, (q + 1) * step), step = ceil(n / world).  Ranks talk
 * through peer memory over NVLink / NVSwitch (a symmetric heap mapped with cudaIpc between processes, direct peer
 * access inside a process); no collective library is called on this path.
 *
 *   build   every rank turns ITS reads' hits into clique pairs, stores each pair straight into the receive buffer
 *           of the rank that owns min(u, v); the owner sorts + deduplicates, sends the reversed copy of every edge
 *           to the owner of max(u, v), and both halves become the owner's CSR rows.  From 2^32 pairs over all
 *           ranks on, the pairs go in rounds (fewer than 2^30 routed to an owner per round) that every owner
 *           merges into its slice of the edge list
 *   peel    one persistent kernel per GPU; a rank logs the unitigs it peels and copies the new part of its log into
 *           every peer (4 bytes per peeled unitig cross a link, whatever its degree); every rank decrements ITS
 *           neighbours of each logged unitig; ranks meet once per cascade generation through flags in peer memory
 *   CORE-A  degree ranks from the summed degree histograms, key ranks from the merged lists of distinct keys
 *
 * This replaces the same reference calls as the single-GPU entry points (src/komb2.cpp:104-132). */
typedef struct kombgpu_comm kombgpu_comm;
typedef struct kombgpu_dist_graph kombgpu_dist_graph;

/* Bootstrap: all-gather `bytes_per_rank` bytes from every rank into `recv` (rank order), blocking, returns 0 on
 * success.  The only service the host has to provide (MPI_Allgather, torch.distributed.all_gather, ...); used
 * to exchange memory handles when the symmetric heap grows, never on the data path. */
typedef int (*kombgpu_allgather_fn)(void *user, const void *send, void *recv, uint64_t bytes_per_rank);

/* Collective over all ranks.  `heap_bytes`: size of a symmetric-heap segment (0 = 512 MiB); the heap grows by
 * segments as needed and is reused across calls.  Every rank must sit on its own GPU of one node. */
int kombgpu_comm_create(kombgpu_ctx *ctx, int rank, int world, kombgpu_allgather_fn allgather, void *user,
                        uint64_t heap_bytes, kombgpu_comm **out);
/* The ranks of ONE process: call from `world` host threads, one per rank, each with its own context, all passing
 * the address of the same pointer variable (initially NULL) as `group_slot`; the bootstrap is built in.  Ranks on
 * distinct GPUs use peer access; all ranks on one GPU is accepted as an emulation mode for tests (the ranks then
 * never wait for one another on the device: exchanges are done by the host threads and the peel runs every rank's
 * share inside one cooperative grid). */
int kombgpu_comm_create_local(kombgpu_ctx *ctx, int rank, int world, void **group_slot, uint64_t heap_bytes,
                              kombgpu_comm **out);
void kombgpu_comm_destroy(kombgpu_comm *comm);
/* A rank of a one-process group whose host code failed: the ranks waiting for it in a collective return
 * KOMBGPU_ESTATE instead of waiting for ever.  (Between processes a missing rank trips the 30 s watchdogs.) */
int kombgpu_comm_abort(kombgpu_comm *comm);
int kombgpu_comm_info(const kombgpu_comm *comm, int *rank, int *world, int *same_device, uint64_t *heap_bytes);

typedef struct kombgpu_dist_stats {
    uint64_t n_hits_local;      /* hits this rank passed in                                     */
    uint64_t n_pairs_local;     /* clique pairs this rank emitted (or pairs passed in)          */
    uint64_t n_pairs_received;  /* pairs routed to this rank (before dedup)                     */
    uint64_t n_fwd_local;       /* edges (u < v) whose u this rank owns                         */
    uint64_t n_directed_local;  /* CSR entries of the local rows                                */
    uint64_t n_edges_global;    /* E                                                            */
    uint64_t n_messages_sent;   /* peel: unitig ids this rank copied into peers' logs           */
    uint64_t n_messages_recv;   /* peel: unitig ids other ranks logged here                     */
    uint32_t n_global, v_lo, n_local;
    int32_t max_degree;         /* global                                                       */
    int32_t max_coreness;       /* global, -1 before the peel                                   */
    uint32_t peel_levels;       /* non-empty levels                                             */
    uint32_t peel_subrounds;    /* cross-rank exchange steps of the peel (all levels)           */
    uint32_t peel_solo_subrounds; /* of those, walked by one CTA on this GPU (thin cascades)    */
    float ms_build, ms_peel, ms_corea;   /* CUDA-event times on this rank                       */
    float ms_build_route, ms_build_sort, ms_build_csr;
    uint32_t peel_async;        /* which peel ran: 0 log-based (ranks meet once per cascade generation), 1 asynchronous
                                   (ranks meet once per level), 2 replicated (small graph: every rank peels all of it) */
} kombgpu_dist_stats;

/* Stage 1..3 over all ranks, collective.  Inputs are device pointers on the rank's device: the hits of THIS
 * rank's reads (both mates, global unitig ids; a read's hits must all be on one rank), or this rank's share of an
 * edge list.  Results stay on the device until fetched.
 * Limits per rank: n_hits < 2^32, distinct (read, unitig) hits < 2^31, edges whose u it owns (n_fwd_local) < 2^32
 * and adjacency entries of its rows (n_directed_local) < 2^32 (KOMBGPU_EINVAL otherwise).  The clique pairs, those a
 * rank emits (or passes in) and those routed to it, are not limited: from 2^32 pairs over all ranks on they are
 * emitted, routed, sorted and merged in rounds, so a rank holds one round of them.  The results do not depend on
 * the rounds.  When one rank fails, every rank returns an error (the failing rank its own) and the contexts and
 * the communicator stay usable. */
int kombgpu_dist_build_hits_dev(kombgpu_comm *comm, const uint32_t *read_key_dev, const uint32_t *unitig_dev,
                                uint64_t n_hits, uint32_t n_vertices_global, kombgpu_dist_graph **out);
int kombgpu_dist_build_pairs_dev(kombgpu_comm *comm, const uint32_t *u_dev, const uint32_t *v_dev, uint64_t n_pairs,
                                 uint32_t n_vertices_global, kombgpu_dist_graph **out);
/* The same with HOST pointers (the rank's share is uploaded first): for hosts without CUDA headers (komb2). */
int kombgpu_dist_build_hits(kombgpu_comm *comm, const uint32_t *read_key, const uint32_t *unitig, uint64_t n_hits,
                            uint32_t n_vertices_global, kombgpu_dist_graph **out);
int kombgpu_dist_build_pairs(kombgpu_comm *comm, const uint32_t *u, const uint32_t *v, uint64_t n_pairs,
                             uint32_t n_vertices_global, kombgpu_dist_graph **out);
int kombgpu_dist_coreness(kombgpu_dist_graph *g);               /* igraph_coreness over all ranks */
int kombgpu_dist_corea(kombgpu_dist_graph *g, int key_mode);    /* CoreA::getAnomalyScore over all ranks */
void kombgpu_dist_graph_destroy(kombgpu_dist_graph *g);

int kombgpu_dist_graph_stats(const kombgpu_dist_graph *g, kombgpu_dist_stats *out);
/* This rank's slice to the host: degree / coreness / score of unitigs [v_lo, v_lo + n_local); any pointer may be
 * NULL. */
int kombgpu_dist_graph_results(const kombgpu_dist_graph *g, int32_t *degree, int32_t *coreness, double *score);
/* This rank's slice of the canonical edge list (the slices of ranks 0, 1, ... concatenate to the global sorted
 * list): u[n_fwd_local], v[n_fwd_local], mult[n_fwd_local]; any pointer may be NULL. */
int kombgpu_dist_graph_edges(const kombgpu_dist_graph *g, uint32_t *u, uint32_t *v, uint32_t *mult);
/* The same slice in CSR form: fwd_ptr[n_local + 1] (edge i has source v_lo + x where fwd_ptr[x] <= i < fwd_ptr[x+1])
 * and v[n_fwd_local]. */
int kombgpu_dist_graph_edges_csr(const kombgpu_dist_graph *g, uint64_t *fwd_ptr, uint32_t *v);
/* Device pointers of the rank's arrays (valid until destroy); any out-pointer may be NULL.  row_ptr / col come
 * back NULL: a rank keeps its adjacency grouped by neighbour for the peel, not as CSR rows. */
int kombgpu_dist_graph_device_arrays(const kombgpu_dist_graph *g, const uint64_t **row_ptr, const uint32_t **col,
                                     const uint64_t **edges_packed, const int32_t **degree, const int32_t **coreness,
                                     const double **score);
/* Global scalars of CombineCoreA::run: max coreness and max CORE-A score (every rank gets the same values). */
int kombgpu_dist_graph_summary(const kombgpu_dist_graph *g, int32_t *max_coreness, double *max_score);

/* The maximal core of the WHOLE partitioned graph and the trussness of its edges: what kombgpu_graph_max_core_truss
 * computes on one GPU, with the same results bit for bit, on every rank.  Collective; needs kombgpu_dist_coreness
 * (KOMBGPU_ESTATE otherwise, on every rank, before any rank waits for another).  Every rank pulls the coreness of
 * the unitigs the other ranks own and their slices of the maximal core's edges, then computes the trussness of the
 * whole maximal core itself: the maximal core has to fit one GPU and hold fewer than 2^32 edges (KOMBGPU_EINVAL on
 * every rank otherwise); the whole graph need not.  When a rank fails, every rank returns an error.  Computed once
 * per graph, cached; the results are held by every rank. */
int kombgpu_dist_max_core_truss(kombgpu_dist_graph *g, uint32_t *n_core_vertices, uint64_t *n_core_edges,
                                int32_t *max_trussness, uint32_t *n_truss_vertices);
/* Local, not collective: the whole result on any rank, as kombgpu_graph_max_core_edges (original unitig ids, u < v,
 * ascending, n_core_edges entries each) and kombgpu_graph_truss_vertices (ascending, n_truss_vertices entries). */
int kombgpu_dist_max_core_edges(const kombgpu_dist_graph *g, uint32_t *u, uint32_t *v, int32_t *trussness);
int kombgpu_dist_truss_vertices(const kombgpu_dist_graph *g, uint32_t *vids);
/* The densest k-core of the WHOLE partitioned graph, as kombgpu_graph_densest_core (same level, sizes and density,
 * same tie rule: equal density goes to the larger block) on every rank.  Collective; needs kombgpu_dist_coreness.
 * The ranks sum their histograms of unitigs per coreness and of edges per min(core(u), core(v)). */
int kombgpu_dist_densest_core(kombgpu_dist_graph *g, int32_t *k_star, uint32_t *n_vertices, uint64_t *n_edges,
                              double *density);
/* The densest BLOCK of the WHOLE partitioned graph, as kombgpu_graph_densest_block (the same passes, sizes, weight
 * sum and density; with weights whose partial sums are exact, such as multiples of a power of two, bit for bit).
 * `weight`: this rank's slice, n_local host doubles >= 0 for unitigs [v_lo, v_lo + n_local), or NULL (weights 0);
 * use_scores != 0 for the graph's own CORE-A scores (needs kombgpu_dist_corea, KOMBGPU_ESTATE otherwise).  eps and
 * use_scores must be the same on every rank.  member (optional): this rank's slice, n_local bytes.  The scalars are
 * global: every rank gets the same values.  Collective; needs only the build; nothing is cached.  The passes are
 * driven by the host: every rank marks its own unitigs, the ranks exchange what they removed (4 bytes per removed
 * unitig cross a link) and every rank lowers the degrees of its own survivors.  The arguments are checked before the
 * first pass: a bad one on any rank gives KOMBGPU_EINVAL there (an eps that differs between the ranks: on every rank)
 * and an error on every other rank.  Any later failure on a rank also makes every rank return an error.  The graph and
 * the communicator stay usable. */
int kombgpu_dist_densest_block(kombgpu_dist_graph *g, const double *weight, int use_scores, double eps,
                               uint32_t *n_vertices, uint64_t *n_edges, double *weight_sum, double *density,
                               uint32_t *n_passes, uint8_t *member);

/* SAM text -> hits over the ranks (kombgpu_sam_parse's token rules, unitig numbering and error messages).  Rank q
 * uploads and parses only the lines that START in bytes [cut_q, cut_{q+1}) of every input, cut_q = the first line
 * start at or after floor(size * q / world) (a line is never split; a slice may be empty).  Every string goes to the
 * rank picked by a fixed-seed hash of its bytes, which interns it by its BYTES (a 64-bit collision rebuilds the table
 * with another seed).  The unitig ids are those of kombgpu_sam_parse on the same inputs: names in order of their
 * first occurrence, every @SQ record before every hit, each group in (input, byte offset) order, names with at least
 * one hit only.  Read ids are unique over the ranks but do NOT follow first appearance: rank q's keys take ids
 * [q * stride, q * stride + n), and all hits of a read, from both mates, end up on that rank (what
 * kombgpu_dist_build_hits_dev needs).  A malformed line anywhere gives KOMBGPU_EINVAL on every rank with the message
 * kombgpu_sam_parse gives (the earliest malformed line in (input, line) order); any other failure on one rank makes
 * every rank return an error.  Limits: fewer than 2^30 lines in a rank's slices, 2^32 routed hits per rank, 2^32 - 1
 * distinct names and keys per rank that interns them, and read ids below 2^32 (KOMBGPU_EINVAL otherwise).  The contexts
 * and the communicator stay usable after an error. */
typedef struct kombgpu_dist_hits kombgpu_dist_hits;
/* Collective.  Every rank passes the same inputs (mate 1 first).  Within one process the pointers may be shared.
 * Between processes, each process maps the files itself. */
int kombgpu_dist_sam_parse(kombgpu_comm *comm, const char *const *texts, const uint64_t *sizes, int n_files,
                           kombgpu_dist_hits **out);
void kombgpu_dist_hits_destroy(kombgpu_dist_hits *h);
/* this rank's hits after routing; global hits, reads, unitigs (= vertices), terminated lines; any pointer may be NULL */
int kombgpu_dist_hits_counts(const kombgpu_dist_hits *h, uint64_t *n_hits_local, uint64_t *n_hits_global,
                             uint32_t *n_reads_global, uint32_t *n_unitigs, uint64_t *n_lines_global);
/* Names of the vertices [v_lo, v_lo + n_local) of the unitig-range partition (step = ceil(n / world), the same
 * partition as kombgpu_dist_graph), as (input, offset inside that input, length); file may be NULL. */
int kombgpu_dist_hits_names(const kombgpu_dist_hits *h, uint32_t *file, uint64_t *offset, uint32_t *len);
/* this rank's routed hits to the host, n_hits_local each; either pointer may be NULL */
int kombgpu_dist_hits_download(const kombgpu_dist_hits *h, uint32_t *read_key, uint32_t *unitig);
int kombgpu_dist_hits_device_arrays(const kombgpu_dist_hits *h, const uint32_t **read_key_dev, const uint32_t **unitig_dev);
/* CUDA-event times of the upload, the parse, the interning and the routing on this rank, and the hash seeds tried */
int kombgpu_dist_hits_timing(const kombgpu_dist_hits *h, float *ms_upload, float *ms_parse, float *ms_intern,
                             float *ms_route, int *hash_rounds);
/* kombgpu_dist_build_hits_dev on the rank's routed hits, with n_vertices_global = n_unitigs.  Collective. */
int kombgpu_dist_build_graph_hits(const kombgpu_dist_hits *h, kombgpu_dist_graph **out);

/* This rank's slice of the output files, formatted on its device: the slices of ranks 0, 1, ... concatenate to
 * exactly the bytes kombgpu_graph_format gives for the same graph on one GPU.  EDGELIST: the rank's slice of the
 * canonical edge list (needs the build); KCORE: rows v_lo .. v_lo + n_local - 1, rank 0's slice starting with the
 * header even when the graph is empty (needs kombgpu_dist_coreness and the kombgpu_dist_hits the graph was built
 * from: the parse leaves every name's bytes on the rank that owns its vertex); COREA: the same rows (needs
 * kombgpu_dist_corea).  Local, NOT collective: a rank formats and fetches when it likes and waits for no other.
 * KOMBGPU_ESTATE for a file whose stage has not run, or a fetch before the format; KOMBGPU_EINVAL for `which` out of
 * range or a KCORE names handle that is missing or belongs to another communicator or partition.  The text is
 * cached in the graph until it is destroyed; fetch and wait work as kombgpu_graph_format_fetch / _wait. */
int kombgpu_dist_graph_format(kombgpu_dist_graph *g, int which, const kombgpu_dist_hits *names, uint64_t *bytes);
int kombgpu_dist_graph_format_fetch(kombgpu_dist_graph *g, int which, char *dst, int async);
int kombgpu_dist_graph_format_wait(kombgpu_dist_graph *g);

/* The unitig FASTA over the ranks: the rules of the single-GPU "unitig FASTA" section above (records, names, join, fence,
 * extraction), with the same results and the same error messages (record numbers, byte offsets and vertex ids are
 * global).  Rank q uploads and indexes only bytes [cut_q, cut_{q+1}) of the file, cut_q = the first record start at or
 * after floor(size * q / world) (cut_0 = 0: bytes before the first record lie in rank 0's slice; a record is never split;
 * a slice may be empty).  Record names and vertex names meet on the rank a fixed-seed hash of their bytes picks, so no
 * GPU holds the whole file, all names or all scores, and nothing of their size passes through the host.  The
 * extraction slices of ranks 0, 1, ... concatenate to exactly the bytes kombgpu_fasta_extract gives on one GPU for the
 * same file, names and mask.  Every call but _counts, _extract_fetch and _timing is collective.  A malformed file, a
 * selected vertex without a record or a bad argument on one rank gives an error on every rank (KOMBGPU_EINVAL with the
 * single-GPU message where one GPU would give it); the contexts, the communicator and the graph stay usable. */
typedef struct kombgpu_dist_fasta kombgpu_dist_fasta;
/* Every rank passes the same bytes of one FASTA file (within one process the pointer may be shared). */
int kombgpu_dist_fasta_load(kombgpu_comm *comm, const char *text, uint64_t size, kombgpu_dist_fasta **out);
void kombgpu_dist_fasta_destroy(kombgpu_dist_fasta *fa);
/* records in this rank's slice, records of the file, first global record id and byte range of the slice; any may be NULL */
int kombgpu_dist_fasta_counts(const kombgpu_dist_fasta *fa, uint32_t *n_records_local, uint32_t *n_records_global,
                              uint32_t *rec_lo, uint64_t *byte_lo, uint64_t *byte_hi);
/* vertex -> record for this rank's vertices: the names of the kombgpu_dist_hits the graph was built from (its unitigs
 * [v_lo, v_lo + n_local)), or a packed host table of n_local names (n_local + 1 offsets, as kombgpu_fasta_join_names);
 * the ranks' vertices follow one another in rank order.  *n_missing: vertices without a record over ALL ranks. */
int kombgpu_dist_fasta_join_hits(kombgpu_dist_fasta *fa, const kombgpu_dist_hits *names, uint32_t *n_missing);
int kombgpu_dist_fasta_join_names(kombgpu_dist_fasta *fa, const char *bytes, const uint64_t *offsets, uint32_t n_local,
                                  uint32_t *n_missing);
/* mask: this rank's n_local host bytes (of its last join).  *bytes: size of THIS rank's slice of the output, which only
 * the rank holding the file's last record ends with the '\n' an unterminated selected last record gets. */
int kombgpu_dist_fasta_extract(kombgpu_dist_fasta *fa, const uint8_t *mask, uint32_t n_local, uint64_t *bytes);
int kombgpu_dist_fasta_extract_fetch(kombgpu_dist_fasta *fa, char *dst);   /* local */
/* CUDA-event times on this rank (they include the waits for the other ranks) and the kernels it launched */
int kombgpu_dist_fasta_timing(const kombgpu_dist_fasta *fa, float *ms_upload, float *ms_index, float *ms_join,
                              float *ms_extract, uint64_t *kernel_launches);
/* The IQR fence on CORE-A over the scores of ALL ranks (needs kombgpu_dist_corea, KOMBGPU_ESTATE otherwise): q1, q3,
 * fence and n_selected are global and bit-equal to kombgpu_graph_anomalous on one GPU; member (optional) is this rank's
 * n_local bytes.  A radix select over the ranks finds the order statistics: no score crosses a link.  Collective. */
int kombgpu_dist_anomalous(kombgpu_dist_graph *g, double whisker, double *q1, double *q3, double *fence,
                           uint32_t *n_selected, uint8_t *member);

int kombgpu_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* KOMBGPU_H */
