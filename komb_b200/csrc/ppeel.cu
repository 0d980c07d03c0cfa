// ppeel.cu — stage 2 over the ranks of a communicator: k-core peel of a graph partitioned by unitig-id range, driven
// entirely from the device.
//
// Replaces igraph_coreness (src/graph.cpp:463) like peel.cu does on one GPU; the result is the same unique
// function of the graph, so it is bit-exact whatever the partition.
//
// One persistent kernel per GPU.  Every rank owns the working degrees of its own unitigs and nobody else touches
// them.  What travels between the GPUs is the FRONTIER, not the decrements: when a rank peels unitigs it appends
// their ids to its LOG, and the new part of the log is copied into every peer's copy of that log (peer memory over
// NVLink; the log of a rank holds each of its unitigs at most once, so it has a fixed size and is never reused).
// Every rank then walks, for each newly logged unitig x of ANY rank, the list of its own unitigs adjacent to x
// (pbuild.cu keeps the local adjacency grouped by neighbour) and decrements them in place.  Per peeled unitig four
// bytes cross a link, whatever its degree; no atomics on shared counters per edge, no per-edge messages.
//
// The peel advances in SUB-ROUNDS, one per cascade generation:
//   [scan]     first sub-round of a level k: local unitigs with degree == k are logged, the alive list is compacted,
//              the smallest surviving degree is noted (empty levels are skipped with it)
//   publish    copy the new part of the own log to every peer (log slots are written once and valid when they differ
//              from an EMPTY marker, so the copy needs no fence and no acknowledgement before it is announced)
//   exchange   ONE meeting of all ranks: each stores, in every peer's control words, the length of its log and its
//              pending work, tagged with the sub-round number, and waits for the same from every peer (flags in peer
//              memory; no host, no collective library)
//   walk       for every newly logged unitig of every rank: decrement the local neighbours; a decrement that takes a
//              degree to k logs that unitig (coreness k) for the next sub-round
// A level ends when no rank logged anything and no slices are pending.  Two things keep a sub-round cheap when
// cascades are thin (hundreds of dependent generations of a few unitigs each, the usual shape of a collapsing core):
// a rank whose share of the sub-round is small runs it SOLO, on CTA 0 alone, while its other CTAs wait on a local
// word -- no grid-wide barrier on the critical path -- and neighbour lists longer than kSliceLen are cut into slices
// that the whole grid shares in the next sub-round.
//
// Ranks that share one device (tests) run inside ONE cooperative grid, a group of CTAs per rank: kernels of
// different ranks must never wait for one another on the same GPU.
#include <cooperative_groups.h>

#include <cstdio>
#include <cstdlib>

#include "prank.cuh"

namespace kg {
namespace {

constexpr int kPThreads = 512;
constexpr int kPWarps = kPThreads / 32;
constexpr int kPU = 4;                       // independent edge chains per lane
constexpr uint32_t kSliceLen = 2048;         // neighbour lists longer than this are cut into slices of this many entries
constexpr uint32_t kSoloWalk = 96;           // a sub-round with at most this many unitigs to walk (and no slices) runs on CTA 0 alone
constexpr unsigned long long kSoloEdges = 8192;
constexpr uint32_t kSoloCopy = 1024;         // a publish of at most this many ids is done by the leader warp alone
constexpr uint32_t kStage = 2048;            // discoveries a CTA collects in shared memory before one append to the log
constexpr int kScanItems = 4;
// The leader CTA of a rank may run ahead of its other CTAs while sub-rounds are SOLO; its decisions are kept in a
// ring indexed by the sub-round number, and every kPlanSync sub-rounds all CTAs of the rank meet, so the lead
// stays below the ring size.
constexpr int kPlanRing = 256;
constexpr uint32_t kPlanSync = 64;

enum : uint32_t { kCopyFull = 1, kWalkFull = 2, kFlagLevelOver = 4, kFlagDone = 8 };

// control words, one block per rank in symmetric memory: w[src][i] is written by rank src
//   0: length of src's log   1: slices pending at src   2: smallest surviving degree at src
struct PeelCtl {
    unsigned long long w[kMaxRanks][4];
};

struct PRankState {
    unsigned long long bar_count, bar_gen;      // barrier of this rank's CTAs
    unsigned long long plan_a[kPlanRing], plan_b[kPlanRing];   // leader -> CTAs: (sub-round << 8) | flags, slot = sub-round % ring
    int32_t k_next[kPlanRing];                  // level of the next sub-round when plan_b says the level is over
    unsigned long long log_hi[kMaxRanks];       // entries of rank q's log that have arrived here
    unsigned long long log_lo[kMaxRanks];       // ... and that have been walked
    unsigned long long n_visited;               // adjacency entries visited (statistics)
    uint32_t log_cnt;                           // length of the own log (appended by scan and walk)
    uint32_t published;                         // ... of which copied to the peers
    uint32_t slice_cnt[2];
    uint32_t alive_out[2];                      // survivors written by a scan (slot = index of the list it wrote)
    int32_t local_min;
    int32_t max_core;
    uint32_t levels, subrounds, solo_subrounds;
    uint32_t error;                             // kErr*
    // where the leader thread's time goes (ns): 0 scan + barrier, 1 plan A, 2 publish copy (+ barrier), 3 wait for the
    // peers, 4 exchange, 5 walk (+ barrier), 6 full publishes, 7 full walks
    unsigned long long prof_ns[8];
    uint32_t full_copy, full_walk;
};

struct PRank {
    uint32_t n_local, v_lo, n_global;
    int world, rank;
    uint32_t ctas;                              // CTAs that work for this rank
    const uint32_t *nbr_ptr;                    // [n_global + 1]
    const uint32_t *nbr;                        // local ids
    int32_t *deg;                               // working degrees (never clamped: only ever decremented)
    int32_t *core;
    uint32_t *alive[2];
    uint64_t *slices[2];                        // first_entry << 12 | (length - 1), length <= kSliceLen
    uint32_t slice_cap;
    uint32_t log_cap;                           // entries per log (the largest n_local)
    PeelCtl *ctl_local;
    PeelCtl *ctl_peer[kMaxRanks];
    uint32_t *log_local[kMaxRanks];             // this rank's copy of rank q's log (q == rank: the log itself)
    uint32_t *log_peer[kMaxRanks];              // rank p's copy of THIS rank's log (peer memory)
    PRankState *st;
};

// discoveries of a CTA are collected in shared memory and appended to the rank's log with ONE atomic per flush
struct Stage {
    uint32_t n;
    uint32_t base;
    uint32_t ids[kStage];
    unsigned long long src_lo[kMaxRanks], src_cnt[kMaxRanks];   // walk stage: the fresh part of every rank's log
};

__device__ __forceinline__ void stage_flush(const PRank &R, PRankState *st, Stage &sg) {   // all threads of the CTA
    __syncthreads();
    const uint32_t n = min(sg.n, kStage);
    __syncthreads();   // everyone has read the count before a fast warp's next batch can add to it
    if (n) {
        if (threadIdx.x == 0) sg.base = atomicAdd(&st->log_cnt, n);
        __syncthreads();
        const uint32_t base = sg.base;
        uint32_t *log = R.log_local[R.rank];
        for (uint32_t i = threadIdx.x; i < n; i += kPThreads) {
            if (base + i < R.log_cap) log[base + i] = sg.ids[i];
            else atomicCAS(&st->error, 0u, (uint32_t)kErrFull);
        }
        __syncthreads();
        if (threadIdx.x == 0) sg.n = 0;
        __syncthreads();
    }
}

// found lanes: coreness k, logged (global id).  Warp-aggregated append to the CTA's stage; when the stage is full the
// excess goes straight to the log (rare: a flush follows every batch).
__device__ __forceinline__ void discover(const PRank &R, PRankState *st, Stage &sg, uint32_t found_mask, bool found, uint32_t loc, int32_t k) {
    if (found_mask == 0) return;
    const uint32_t lane = lane_id();
    const uint32_t cnt = (uint32_t)__popc(found_mask);
    uint32_t pos = 0;
    if (lane == 0) pos = atomicAdd(&sg.n, cnt);
    pos = __shfl_sync(kFullMask, pos, 0) + __popc(found_mask & lanemask_lt());
    if (found) {
        R.core[loc] = k;
        if (pos < kStage) {
            sg.ids[pos] = R.v_lo + loc;
        } else {
            const uint32_t at = atomicAdd(&st->log_cnt, 1u);
            if (at < R.log_cap) R.log_local[R.rank][at] = R.v_lo + loc;
            else atomicCAS(&st->error, 0u, (uint32_t)kErrFull);
        }
    }
}

// walk entries [0, total) of a batch of neighbour lists, one list per lane (first entry, excl prefix of the lengths)
__device__ __forceinline__ void walk_lists(const PRank &R, PRankState *st, Stage &sg, uint32_t first, uint32_t excl, uint32_t total,
                                           int32_t k) {
    const uint32_t lane = lane_id();
    const bool look_first = total > 32u * kPU;
    for (uint32_t base = 0; base < total; base += 32u * kPU) {
        uint32_t u[kPU];
        int32_t d[kPU];
#pragma unroll
        for (int t = 0; t < kPU; ++t) {
            const uint32_t e = base + t * 32u + lane;
            u[t] = 0xffffffffu;
            if (base + t * 32u >= total) continue;   // warp-uniform
            uint32_t j = 0;   // owner list: the last lane j with excl[j] <= e
#pragma unroll
            for (uint32_t s = 16; s > 0; s >>= 1) {
                const uint32_t x = __shfl_sync(kFullMask, excl, (j + s) & 31u);
                if (j + s < 32u && x <= e) j += s;
            }
            const uint32_t ex_j = __shfl_sync(kFullMask, excl, j);
            const uint32_t f_j = __shfl_sync(kFullMask, first, j);
            if (e < total) u[t] = R.nbr[f_j + (e - ex_j)];
        }
        // degrees never go up and are never clamped: the decrement that takes a degree from k + 1 to k owns the unitig.
        // Thin batches decrement without looking (one round trip less on a cascade's critical path); wide ones look first
        // (no atomic on unitigs that are already gone).
#pragma unroll
        for (int t = 0; t < kPU; ++t)
            d[t] = u[t] == 0xffffffffu ? INT32_MIN : (look_first ? __ldcg(&R.deg[u[t]]) : INT32_MAX);
#pragma unroll
        for (int t = 0; t < kPU; ++t) d[t] = d[t] > k ? atomicSub(&R.deg[u[t]], 1) : INT32_MIN;
#pragma unroll
        for (int t = 0; t < kPU; ++t) {
            if (base + t * 32u >= total) continue;
            const bool found = d[t] == k + 1;
            discover(R, st, sg, __ballot_sync(kFullMask, found), found, u[t], k);
        }
    }
}

// WALK stage for the warps of one CTA (gw: index of this warp among the nw warps that walk for the rank): pending
// slices, then the newly logged unitigs of every rank.  The CTA flushes its stage after every batch.
__device__ __forceinline__ void walk_stage(const PRank &R, PRankState *st, Stage &sg, uint32_t gw, uint32_t nw, uint32_t cur, int32_t k) {
    const uint32_t lane = lane_id(), warp = threadIdx.x >> 5;
    const uint32_t nxt = cur ^ 1u;
    unsigned long long visited = 0;
    // ---- slices (each is one batch of a warp)
    const uint32_t n_sl = __ldcg(&st->slice_cnt[cur]);
    const uint32_t cta_w0 = gw - warp, per_round = nw;   // the warps of a CTA advance together, one batch each per round
    for (uint32_t i0 = cta_w0; i0 < n_sl; i0 += per_round) {
        const uint32_t i = i0 + warp;
        if (i < n_sl) {
            const uint64_t sl = __ldcg(&R.slices[cur][i]);
            const uint32_t len = (uint32_t)(sl & 0xfffu) + 1u;
            walk_lists(R, st, sg, (uint32_t)(sl >> 12), lane == 0 ? 0u : len, len, k);
            visited += lane == 0 ? len : 0u;
        }
        stage_flush(R, st, sg);
    }
    // ---- newly logged unitigs, all sources concatenated
    if (threadIdx.x < kMaxRanks) {
        unsigned long long lo = 0, cnt = 0;
        if ((int)threadIdx.x < R.world) {
            lo = __ldcg(&st->log_lo[threadIdx.x]);
            cnt = __ldcg(&st->log_hi[threadIdx.x]) - lo;
        }
        sg.src_lo[threadIdx.x] = lo;
        sg.src_cnt[threadIdx.x] = cnt;
    }
    __syncthreads();
    unsigned long long total_new = 0;
    for (int q = 0; q < R.world; ++q) total_new += sg.src_cnt[q];
    // unitigs per warp batch: few fresh unitigs are spread over all the warps (a collapsing core peels a few hundred
    // unitigs with hundreds of neighbours each per generation: one list per warp, not 32)
    const uint32_t b = (uint32_t)min(max((total_new + nw - 1) / nw, 1ull), 32ull);
    for (unsigned long long c0 = (unsigned long long)cta_w0 * b; c0 < total_new; c0 += (unsigned long long)per_round * b) {
        const unsigned long long i = c0 + (unsigned long long)warp * b + lane;
        uint32_t first = 0, len = 0;
        if (lane < b && i < total_new) {
            unsigned long long off = i;
            int q = 0;
            while (off >= sg.src_cnt[q]) { off -= sg.src_cnt[q]; ++q; }   // which source's log (i < total_new: q stays < world)
            const uint32_t x = log_read(&R.log_local[q][sg.src_lo[q] + off], st);
            if (x >= R.n_global) {
                atomicCAS(&st->error, 0u, (uint32_t)kErrBadEntry);
            } else {
                first = R.nbr_ptr[x];
                len = R.nbr_ptr[x + 1] - first;
            }
        }
        // long lists are cut into slices that the whole grid walks in the next sub-round
        const uint32_t n_cut = len > kSliceLen ? (len + kSliceLen - 1) / kSliceLen : 0u;
        if (__ballot_sync(kFullMask, n_cut != 0)) {
            const uint32_t inc = warp_incl_scan_add(n_cut);
            const uint32_t tot = __shfl_sync(kFullMask, inc, 31);
            uint32_t pos = 0;
            if (lane == 0) pos = atomicAdd(&st->slice_cnt[nxt], tot);
            pos = __shfl_sync(kFullMask, pos, 0) + (inc - n_cut);
            for (uint32_t s = 0; s < n_cut; ++s) {
                const uint32_t l = min(kSliceLen, len - s * kSliceLen);
                if (pos + s < R.slice_cap) R.slices[nxt][pos + s] = ((uint64_t)(first + s * kSliceLen) << 12) | (uint64_t)(l - 1u);
                else atomicCAS(&st->error, 0u, (uint32_t)kErrFull);
            }
            if (n_cut) len = 0;
        }
        const uint32_t incl = warp_incl_scan_add(len);
        const uint32_t total = __shfl_sync(kFullMask, incl, 31);
        walk_lists(R, st, sg, first, incl - len, total, k);
        visited += lane == 0 ? total : 0u;
        stage_flush(R, st, sg);
    }
    if (lane == 0 && visited) atomicAdd(&st->n_visited, visited);
}

// SCAN stage of level k (all CTAs of the rank): alive unitigs at degree k are logged, survivors compacted
__device__ __forceinline__ void scan_stage(const PRank &R, PRankState *st, uint32_t cta, const uint32_t *alive_src, uint32_t n_alive,
                                           uint32_t *alive_dst, uint32_t *alive_out, int32_t k, uint32_t *s_scan, uint32_t *s_base) {
    const uint32_t tid = threadIdx.x;
    int32_t local_min = INT32_MAX;
    const uint32_t tile = kPThreads * kScanItems;
    uint32_t *log = R.log_local[R.rank];
    for (uint64_t t0 = (uint64_t)cta * tile; t0 < n_alive; t0 += (uint64_t)R.ctas * tile) {
        uint32_t v[kScanItems], flag[kScanItems];
        uint32_t mine = 0;
#pragma unroll
        for (int j = 0; j < kScanItems; ++j) {
            const uint64_t i = t0 + (uint64_t)j * kPThreads + tid;
            flag[j] = 0;
            v[j] = 0;
            if (i < n_alive) {
                v[j] = alive_src ? __ldcg(&alive_src[i]) : (uint32_t)i;
                const int32_t d = __ldcg(&R.deg[v[j]]);
                if (d == k) {
                    R.core[v[j]] = k;
                    flag[j] = 1u;    // logged even at k = 0 (nothing to walk, but the log's length counts the peeled unitigs)
                } else if (d > k) {
                    flag[j] = 0x10000u;
                    local_min = min(local_min, d);
                }
            }
            mine += flag[j];
        }
        uint32_t total = 0;
        const uint32_t ex = block_excl_scan_add<uint32_t, kPThreads>(mine, s_scan, &total);
        if (tid == 0) {
            const uint32_t nf = total & 0xffffu, ns = total >> 16;
            s_base[0] = nf ? atomicAdd(&st->log_cnt, nf) : 0;
            s_base[1] = ns ? atomicAdd(alive_out, ns) : 0;
        }
        __syncthreads();
        uint32_t fpos = s_base[0] + (ex & 0xffffu), spos = s_base[1] + (ex >> 16);
#pragma unroll
        for (int j = 0; j < kScanItems; ++j) {
            if (flag[j] == 1u) {
                if (fpos < R.log_cap) log[fpos] = R.v_lo + v[j];
                else atomicCAS(&st->error, 0u, (uint32_t)kErrFull);
                ++fpos;
            } else if (flag[j]) {
                alive_dst[spos++] = v[j];
            }
        }
        __syncthreads();
    }
    local_min = warp_reduce_min(local_min);
    if (lane_id() == 0 && local_min != INT32_MAX) atomicMin(&st->local_min, local_min);
}

// The leader (warp 0 of the rank's CTA 0) meets the other ranks: publish the counts, wait, decide.
// Lane 0 never stores into peer memory: it is the thread that releases the plan to the rank's other CTAs, and a
// release (or fence) waits for the calling thread's own outstanding stores -- for stores that crossed NVLink that is
// a full round trip.  Lane q + 1 talks to rank q.
__device__ __forceinline__ void leader_exchange(const PRank &R, PRankState *st, uint32_t t, uint32_t cur, int32_t k, bool scanned,
                                                bool copy_here, unsigned long long &peer_log_hi, uint32_t &published) {
    const uint32_t lane = lane_id();
    const int world = R.world;
    const int peer = (int)lane - 1;                 // the rank this lane talks to (lanes 1 .. world)
    const bool has_peer = peer >= 0 && peer < world;
    const unsigned long long tag = (unsigned long long)t << kTagShift;
    unsigned long long log_len = 0, n_slices = 0;
    uint32_t pub_lo = 0;
    int32_t lmin = INT32_MAX;
    if (lane == 0) {
        log_len = __ldcg(&st->log_cnt);
        n_slices = __ldcg(&st->slice_cnt[cur]);
        lmin = __ldcg(&st->local_min);
        st->published = (uint32_t)log_len;
    }
    log_len = __shfl_sync(kFullMask, log_len, 0);
    n_slices = __shfl_sync(kFullMask, n_slices, 0);
    lmin = __shfl_sync(kFullMask, lmin, 0);
    pub_lo = published;          // every lane of the leader warp carries it in a register
    published = (uint32_t)log_len;
    if (copy_here && world > 1 && lane > 0) {
        // a short new part of the log: this warp copies it to the peers itself, then announces it -- no barrier, no fence
        const uint32_t *src = R.log_local[R.rank];
        for (uint32_t i = pub_lo + (lane - 1u); i < (uint32_t)log_len; i += 31u) {
            const uint32_t x = __ldcg(&src[i]);
            for (int p = 0; p < world; ++p)
                if (p != R.rank) R.log_peer[p][i] = x;
        }
    }
    if (has_peer) {
        PeelCtl *dst = R.ctl_peer[peer];
        st_relaxed_sys(&dst->w[R.rank][1], tag | n_slices);
        st_relaxed_sys(&dst->w[R.rank][2], tag | (unsigned long long)(uint32_t)lmin);
        st_relaxed_sys(&dst->w[R.rank][0], tag | log_len);
    }
    // wait for every rank's words of this sub-round
    const unsigned long long t_wait = pglobal_ns();
    unsigned long long w0 = 0, w1 = 0, w2 = (unsigned long long)(uint32_t)INT32_MAX;
    bool failed = false;
    if (has_peer) {
        const PeelCtl *mine = R.ctl_local;
        uint32_t spins = 0;
        while (true) {
            w0 = ld_relaxed_sys(&mine->w[peer][0]);
            w1 = ld_relaxed_sys(&mine->w[peer][1]);
            w2 = ld_relaxed_sys(&mine->w[peer][2]);
            if ((w0 >> kTagShift) == t && (w1 >> kTagShift) == t && (w2 >> kTagShift) == t) break;
            if ((++spins & 1023u) == 0 && (*(volatile uint32_t *)&st->error || pglobal_ns() - t_wait > kPeelWatchdogNs)) { failed = true; break; }
        }
        w0 &= kValMask; w1 &= kValMask; w2 &= kValMask;
    }
    if (lane == 0) st->prof_ns[3] += pglobal_ns() - t_wait;
    if (__ballot_sync(kFullMask, failed)) {
        if (lane == 0) {
            atomicCAS(&st->error, 0u, (uint32_t)kErrPeers);
            st_rel_gpu(&st->plan_b[t % kPlanRing], ((unsigned long long)t << 8) | kFlagDone);
        }
        return;
    }
    // lane 0 records the new log lengths itself (its release of the plan then covers them); the previous lengths live in
    // the registers of the lanes that talk to the peers: nothing is loaded here
    const unsigned long long my_before = peer_log_hi;
    if (has_peer) peer_log_hi = w0;
    unsigned long long g_fresh = 0, g_slices = 0, g_total = 0;
    uint32_t g_min = (uint32_t)INT32_MAX;
    for (int q = 0; q < world; ++q) {
        const unsigned long long hi = __shfl_sync(kFullMask, w0, q + 1);
        const unsigned long long before = __shfl_sync(kFullMask, my_before, q + 1);
        g_slices += __shfl_sync(kFullMask, w1, q + 1);
        g_min = min(g_min, (uint32_t)__shfl_sync(kFullMask, w2, q + 1));
        g_total += hi;
        g_fresh += hi - before;
        if (lane == 0) {
            st->log_lo[q] = before;
            st->log_hi[q] = hi;
        }
    }
    // few fresh unitigs and nothing pending: this rank walks them on CTA 0 alone (their lists are at most kSliceLen long)
    const unsigned long long my_entries = (g_fresh <= kSoloWalk && n_slices == 0) ? 0ull : ~0ull;
    if (lane == 0) {
        uint32_t flags = (my_entries <= kSoloEdges) ? 0u : kWalkFull;
        st->subrounds = t;
        if (scanned && g_fresh) { st->levels += 1; st->max_core = k; }
        if (g_fresh == 0 && g_slices == 0) {
            // nobody logged anything and nothing is pending: the level is over
            flags |= kFlagLevelOver;
            if (g_total >= R.n_global) flags |= kFlagDone;               // every unitig of the graph is in a log
            if (scanned) {
                if (g_min == (uint32_t)INT32_MAX) flags |= kFlagDone;    // nothing alive anywhere
                st->k_next[t % kPlanRing] = (int32_t)g_min;               // the level was empty: skip to the smallest degree
            } else {
                st->k_next[t % kPlanRing] = k + 1;
            }
            st->local_min = INT32_MAX;
        } else if (!(flags & kWalkFull)) {
            st->solo_subrounds += 1;
        }
        st_rel_gpu(&st->plan_b[t % kPlanRing], ((unsigned long long)t << 8) | flags);
    }
}

__global__ void __launch_bounds__(kPThreads, 2) ppeel_kernel(const PRank *ranks, uint32_t ctas_per_rank) {
    __shared__ uint32_t s_scan[kPWarps + 1];
    __shared__ uint32_t s_base[2];
    __shared__ uint32_t s_bcast;
    __shared__ Stage s_stage;
    const PRank R = ranks[blockIdx.x / ctas_per_rank];
    PRankState *st = R.st;
    const uint32_t cta = blockIdx.x % ctas_per_rank;
    const uint32_t tid = threadIdx.x, warp = tid >> 5;
    const bool leader_cta = cta == 0;
    unsigned long long bar_gen = 0;
    uint32_t t = 1;          // sub-round number (tags of zero-initialised control words are 0)
    int32_t k = 0;
    bool scan = true;
    uint32_t cur = 0;        // slice list walked this sub-round
    const uint32_t *alive_src = nullptr;   // nullptr: every local unitig
    uint32_t alive_i = 0;
    uint32_t n_alive = R.n_local;
    if (tid == 0) s_stage.n = 0;
    __syncthreads();
    unsigned long long peer_log_hi = 0;   // leader warp, lane q + 1: length of rank q's log at the last exchange
    uint32_t published = 0;               // leader warp: length of the own log at the last exchange

    const bool prof = leader_cta && tid == 0;
    unsigned long long tp = prof ? pglobal_ns() : 0ull;
#define KG_PROF(slot)                                               \
    if (prof) {                                                     \
        const unsigned long long now_ = pglobal_ns();               \
        st->prof_ns[slot] += now_ - tp;                             \
        tp = now_;                                                  \
    }
    while (true) {
        if (scan) {
            scan_stage(R, st, cta, alive_src, n_alive, R.alive[alive_i], &st->alive_out[alive_i], k, s_scan, s_base);
            rank_barrier(st, R.ctas, bar_gen, false);
            n_alive = __ldcg(&st->alive_out[alive_i]);
            alive_src = R.alive[alive_i];
            alive_i ^= 1u;
            // the other slot was last read two scans ago (every CTA has passed a barrier since): re-arm it for the next scan
            if (leader_cta && tid == 0) st->alive_out[alive_i] = 0;
        } else if ((t % kPlanSync) == 0) {
            rank_barrier(st, R.ctas, bar_gen, false);   // bounds the leader's lead over the other CTAs (plan ring)
        }
        KG_PROF(0);
        // ---- plan A: who copies the new part of the log to the peers
        if (leader_cta && tid == 0) {
            const uint32_t fresh = __ldcg(&st->log_cnt) - __ldcg(&st->published);
            const uint32_t mode = (R.world > 1 && fresh > kSoloCopy) ? kCopyFull : 0u;
            st_rel_gpu(&st->plan_a[t % kPlanRing], ((unsigned long long)t << 8) | mode);
        }
        const uint32_t mode_a = wait_plan<kFlagDone>(&st->plan_a[t % kPlanRing], t, st, &s_bcast);
        if (mode_a & kFlagDone) break;   // watchdog
        KG_PROF(1);
        // ---- publish
        if (mode_a & kCopyFull) {
            publish_stage(R, st, cta * kPThreads + tid, R.ctas * kPThreads);
            rank_barrier(st, R.ctas, bar_gen, false);
            if (prof) { st->full_copy += 1; st->prof_ns[6] += pglobal_ns() - tp; }
        }
        KG_PROF(2);
        // ---- exchange (a short publish is done by the leader warp itself)
        if (leader_cta && warp == 0) leader_exchange(R, st, t, cur, k, scan, !(mode_a & kCopyFull), peer_log_hi, published);
        const uint32_t flags = wait_plan<kFlagDone>(&st->plan_b[t % kPlanRing], t, st, &s_bcast);
        KG_PROF(4);
        // ---- walk
        if (!(flags & kFlagLevelOver)) {
            if (flags & kWalkFull) {
                walk_stage(R, st, s_stage, cta * kPWarps + warp, R.ctas * kPWarps, cur, k);
                rank_barrier(st, R.ctas, bar_gen, false);
                if (prof) { st->full_walk += 1; st->prof_ns[7] += pglobal_ns() - tp; }
            } else if (leader_cta) {
                walk_stage(R, st, s_stage, warp, kPWarps, cur, k);
                __syncthreads();
                if (tid == 0) __threadfence();
                __syncthreads();
            }
            // the slice list that was walked becomes the one the next sub-round's walk appends to
            if (leader_cta && tid == 0) st->slice_cnt[cur] = 0;
            cur ^= 1u;
        }
        KG_PROF(5);
        if ((flags & kFlagDone) || *(volatile uint32_t *)&st->error) break;
        ++t;
        if (t >= (1u << 24) - 2u) { if (tid == 0) atomicCAS(&st->error, 0u, (uint32_t)kErrBarrier); break; }
        if (flags & kFlagLevelOver) {
            k = __ldcg(&st->k_next[(t - 1u) % kPlanRing]);
            scan = true;
        } else {
            scan = false;
        }
    }
#undef KG_PROF
}

}  // namespace

int dist_peel(kombgpu_dist_graph *g, int rc) {
    kombgpu_comm *c = g->comm;
    kombgpu_ctx *ctx = g->ctx;
    const int world = c->world;
    const uint32_t n_local = g->n_local;

    // symmetric: one log per rank (every rank holds a copy of every rank's log) + the control words
    const uint32_t log_cap = g->step;   // the largest n_local
    SymRewind heap{c, sym_mark(c)};
    uint32_t *logs = nullptr;
    PeerPtrs<uint32_t> logs_peers{};
    PeelCtl *ctl = nullptr;
    PeerPtrs<PeelCtl> ctl_peers{};
    rc = first_rc(rc, sym_alloc(c, (size_t)world * log_cap, &logs, &logs_peers));
    rc = first_rc(rc, sym_alloc(c, 1, &ctl, &ctl_peers));

    // per-rank lists and state
    DevBuf<int32_t> work;
    DevBuf<uint32_t> alive_a, alive_b;
    DevBuf<uint64_t> slices_a, slices_b;
    DevBuf<PRankState> state;
    DevBuf<PRank> desc;
    uint32_t ctas_per_rank = 0;
    PRank R{};
    if (rc == KOMBGPU_OK) rc = [&]() -> int {
        KG_CUDA(ctx, cudaMemsetAsync(g->core, 0, (size_t)(n_local ? n_local : 1) * sizeof(int32_t), ctx->stream));
        KG_CUDA(ctx, cudaMemsetAsync(ctl, 0, sizeof(PeelCtl), ctx->stream));
        KG_CUDA(ctx, cudaMemsetAsync(logs, 0xff, (size_t)world * log_cap * sizeof(uint32_t), ctx->stream));   // kLogEmpty
        // every unitig of the graph is walked once here, its list cut into ceil(len / kSliceLen) slices when it is long
        const uint64_t slice_cap64 = g->n_directed / kSliceLen + (uint64_t)g->n_global / 64 + 1024;
        if (slice_cap64 >= 0xffffffffull) return ctx_fail(ctx, KOMBGPU_EINVAL, "partition too large for the slice list");
        KG_ALLOC(ctx, work, n_local);
        KG_ALLOC(ctx, alive_a, n_local);
        KG_ALLOC(ctx, alive_b, n_local);
        KG_ALLOC(ctx, slices_a, slice_cap64);
        KG_ALLOC(ctx, slices_b, slice_cap64);
        KG_ALLOC(ctx, state, 1);
        KG_ALLOC(ctx, desc, kMaxRanks);
        KG_CUDA(ctx, cudaMemcpyAsync(work.p, g->deg, (size_t)n_local * sizeof(int32_t), cudaMemcpyDeviceToDevice, ctx->stream));
        PRankState init{};
        init.local_min = INT32_MAX;
        KG_CUDA(ctx, cudaMemcpyAsync(state.p, &init, sizeof(init), cudaMemcpyHostToDevice, ctx->stream));
        KG_TRY(rank_ctas(ctx, c, ppeel_kernel, kPThreads, 1, &ctas_per_rank));
        R.n_local = n_local; R.v_lo = g->v_lo; R.n_global = g->n_global; R.world = world; R.rank = c->rank; R.ctas = ctas_per_rank;
        R.nbr_ptr = g->nbr_ptr; R.nbr = g->nbr; R.deg = work.p; R.core = g->core;
        R.alive[0] = alive_a.p; R.alive[1] = alive_b.p;
        R.slices[0] = slices_a.p; R.slices[1] = slices_b.p; R.slice_cap = (uint32_t)slice_cap64;
        R.log_cap = log_cap;
        R.ctl_local = ctl;
        for (int q = 0; q < world; ++q) {
            R.ctl_peer[q] = ctl_peers.p[q];
            R.log_local[q] = logs + (size_t)q * log_cap;                         // my copy of rank q's log
            R.log_peer[q] = logs_peers.p[q] + (size_t)c->rank * log_cap;        // rank q's copy of my log
        }
        R.st = state.p;
        return KOMBGPU_OK;
    }();
    // every rank's control words are cleared before anyone publishes into them
    KG_TRY(barrier_rc(c, rc));

    const cudaError_t le = launch_ranks(c, ppeel_kernel, kPThreads, ctas_per_rank, R, desc.p, nullptr);
    if (le != cudaSuccess) rc = ctx_fail(ctx, KOMBGPU_ECUDA, "partitioned peel kernel: %s", cudaGetErrorString(le));
    PRankState fin{};
    if (rc == KOMBGPU_OK) rc = read_back(ctx, state.p, &fin, 1);
    // global figures; also: nobody gives back its logs (at return) while a peer may still be writing
    unsigned long long mine[3] = {fin.error, fin.log_cnt, (unsigned long long)(uint32_t)fin.max_core}, all[kMaxRanks * 3];
    KG_TRY(exchange_rc(c, rc, mine, 3, all));
    uint64_t peeled = 0;
    for (int q = 0; q < world; ++q) {
        if (all[q * 3]) return ctx_fail(ctx, KOMBGPU_EINTERNAL, "partitioned peel: rank %d reports error %llu (%s)", q, all[q * 3], rank_error_text(all[q * 3]));
        peeled += all[q * 3 + 1];
    }
    if (peeled != g->n_global) return ctx_fail(ctx, KOMBGPU_EINTERNAL, "partitioned peel ended with %llu of %u unitigs peeled", (unsigned long long)peeled, g->n_global);
    g->st.max_coreness = fin.max_core;
    g->st.peel_levels = fin.levels;
    g->st.peel_subrounds = fin.subrounds;
    g->st.peel_solo_subrounds = fin.solo_subrounds;
    g->st.n_messages_sent = (uint64_t)fin.log_cnt * (uint64_t)(world - 1);   // ids copied to peers
    g->st.n_messages_recv = peeled - fin.log_cnt;
    if (getenv("KOMBGPU_DEBUG"))
        fprintf(stderr, "[kombgpu] rank %d ppeel: levels %u subrounds %u (solo walks %u; full copies %u, full walks %u) ctas %u | leader ms: scan %.3f planA %.3f "
                "publish %.3f (full %.3f) exchange %.3f (wait peers %.3f) walk %.3f (full %.3f) | peeled here %u, entries visited %llu\n",
                c->rank, fin.levels, fin.subrounds, fin.solo_subrounds, fin.full_copy, fin.full_walk, ctas_per_rank, fin.prof_ns[0] * 1e-6,
                fin.prof_ns[1] * 1e-6, fin.prof_ns[2] * 1e-6, fin.prof_ns[6] * 1e-6, fin.prof_ns[4] * 1e-6, fin.prof_ns[3] * 1e-6,
                fin.prof_ns[5] * 1e-6, fin.prof_ns[7] * 1e-6, fin.log_cnt, fin.n_visited);
    return KOMBGPU_OK;
}

}  // namespace kg
