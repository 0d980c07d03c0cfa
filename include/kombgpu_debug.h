/*
 * kombgpu_debug.h -- measurement aids of libkombgpu.so.  NOT part of the product ABI (include/kombgpu.h):
 * nothing here replaces anything in the reference; the probes under tools/ and one sort test use them.
 */
#ifndef KOMBGPU_DEBUG_H
#define KOMBGPU_DEBUG_H

#include "kombgpu.h"

#ifdef __cplusplus
extern "C" {
#endif

/* tools/sort_probe.py: sorts n synthetic 64-bit keys with lo_bits random low bits and hi_bits bits at
 * position 32 (random, or non-decreasing when sorted_hi != 0: the shape of hit arrays in read order) on
 * bits [0, lo_bits) + [32, 32 + hi_bits), `reps` times; returns the best time of the sort alone and
 * whether the result is a sorted permutation of the input. */
int kombgpu_debug_sort_u64(kombgpu_ctx *ctx, uint64_t n, int lo_bits, int hi_bits, int sorted_hi, int reps,
                           float *ms_best, int *ok);

/* tools/peel_ab.py, tools/peel_trace*.py: run the k-core peel again on a graph that already holds its
 * coreness (kombgpu_coreness peels once per graph), so one build serves many timed peels. */
int kombgpu_debug_peel_again(kombgpu_graph *g);

/* tests/test_pair_chunks_gpu.py, tools/pair_chunk_probe.py: the number of chunks a graph built from hits or pairs
 * reduced its clique pairs in.  1 is the one-shot path; the chunked path runs when the pairs reach 2^32 or, with
 * KOMBGPU_PAIR_CHUNK=<pairs> set, when they exceed that many (the chunk size).  0 for a graph adopted from a CSR. */
int kombgpu_debug_build_chunks(const kombgpu_graph *g, uint32_t *n_chunks);

/* tests/test_dist_pair_chunks_gpu.py, tools/dist_pair_chunk_probe.py: the number of rounds a multi-GPU build emitted,
 * routed and reduced its clique pairs in.  1 is the one-shot path; the rounds run when the pairs of all ranks reach
 * 2^32 or, with KOMBGPU_PAIR_CHUNK=<pairs> set, when some rank's pairs exceed that many (the pairs per rank and round). */
int kombgpu_debug_dist_build_rounds(const kombgpu_dist_graph *g, uint32_t *n_rounds);

/* tools/dist_truss_probe.py: the CUDA-event split of this rank's last kombgpu_dist_max_core_truss -- the gather of the
 * coreness, the selection of the maximal core with the gather of the edge slices, and the truss peel. */
int kombgpu_debug_dist_truss_timing(const kombgpu_dist_graph *g, float *ms_core_gather, float *ms_slice_gather,
                                    float *ms_truss);

#ifdef __cplusplus
}
#endif
#endif /* KOMBGPU_DEBUG_H */
