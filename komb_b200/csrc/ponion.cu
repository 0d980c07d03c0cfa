// ponion.cu — onion layers (onion.cu) over the ranks of a communicator: a peel of the partitioned graph whose steps are
// exactly the layers of the synchronous peel, bit-equal to one GPU whatever the partition.
//
// One persistent kernel per GPU, driven from the device, built like the log-based peel (ppeel.cu): every rank owns
// the working degrees of its own unitigs and nobody else touches them; a rank appends the ids it removes to its LOG,
// copies the new part of the log into every peer's copy through peer memory, and walks, for every id logged by any
// rank in the previous step, the list of its own unitigs adjacent to that id (nbr_ptr / nbr) and decrements them.
//
// The layer rule is onion.cu's: degree-0 unitigs form layer 1 when there are any; a level k starts with a SCAN that
// logs the local unitigs at degree k as the level's first layer; while layer l is walked, the decrement that takes a
// degree from k + 1 to k logs that unitig into layer l + 1 with coreness k; degrees are never clamped.
//
// What ppeel.cu gives up for speed the onion needs: a step of ppeel walks long lists one sub-round late (slices) and
// lets its leader CTA run ahead, so its sub-rounds are not layers.  Here a step walks every id of layer l from every
// rank AND all slices of the long lists among them -- lists first, a barrier of the rank's CTAs, then the slices --
// and only then publishes and meets the other ranks.  So every decrement caused by layer l has landed on its owner
// before any rank forms layer l + 1.  Each step ends with ONE meeting of all ranks (control words in peer memory,
// tagged with the step number): each rank's log length and, at scan steps, its smallest surviving degree.  From them
// every rank derives the same size of the layer just formed, whether the level is over, and the next k (the global
// minimum of the survivors' degrees, so empty levels are skipped), and the number of the last non-empty layer.
//
// A rank whose share of a walk step is small (at most kSoloIds ids over all ranks and kSoloEdges local entries) runs
// it on CTA 0 alone, while its other CTAs wait for the next plan: a chain of thin layers costs no barrier of the
// rank's CTAs.  Ranks that share one device (tests) run inside ONE cooperative grid, a group of CTAs each.
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "kombgpu_debug.h"
#include "prank.cuh"

namespace kg {
namespace {

constexpr int kOThreads = 512;
constexpr int kOWarps = kOThreads / 32;
constexpr int kOUnroll = 4;                  // independent nbr -> atomic chains per thread
constexpr int kOScanItems = 4;
constexpr uint32_t kOSliceLen = 2048;        // in a step on all CTAs, lists longer than this are cut into slices
constexpr uint32_t kSoloIds = kOThreads;     // a walk step with at most this many ids over all ranks ...
constexpr uint32_t kSoloEdges = 16384;       // ... and at most this many local entries runs on CTA 0 alone
// CTA 0 may run ahead of the rank's other CTAs while steps are solo: the plans are kept in a ring indexed by the step
// number, and every kOPlanSync steps all CTAs of the rank meet, so the lead stays below the ring size.
constexpr int kOPlanRing = 256;
constexpr uint32_t kOPlanSync = 64;

enum : uint32_t { kPlanWalk = 1, kPlanFull = 2, kPlanDone = 4 };   // the next step: a walk (else a scan), on all CTAs, or none

// control words, one block per rank in symmetric memory: w[t & 1][src][i] is written by rank src at step t
//   0: length of src's log   1: smallest surviving degree at src (scan steps)
// Two parities: a rank can be one step ahead of a peer that has not read its words yet, never two.
struct OnionCtl {
    unsigned long long w[2][kMaxRanks][2];
};

struct ORankState {
    unsigned long long bar_count, bar_gen;      // barrier of this rank's CTAs
    unsigned long long plan[kOPlanRing];        // CTA 0 -> CTAs: (step << 8) | flags of the NEXT step, slot = step % ring
    int32_t plan_k[kOPlanRing];                 // ... its level
    uint32_t plan_layer[kOPlanRing];            // ... and the number of the last non-empty layer before it
    unsigned long long log_lo[kMaxRanks];       // the ids of rank q walked by the next walk step: its log [log_lo, log_hi)
    unsigned long long log_hi[kMaxRanks];
    uint32_t log_cnt;                           // length of the own log
    uint32_t published;                         // ... of which copied to the peers
    uint32_t slice_cnt;
    uint32_t alive_out[2];                      // survivors written by a scan (slot = index of the list it wrote)
    int32_t local_min;
    uint32_t n_layers, levels, meetings, solo_steps;
    uint32_t error;                             // kErr*
};

struct ORank {
    uint32_t n_local, v_lo, n_global;
    int world, rank;
    uint32_t ctas;                              // CTAs that work for this rank
    const uint32_t *nbr_ptr;                    // [n_global + 1]
    const uint32_t *nbr;                        // local ids
    int32_t *deg;                               // working degrees (never clamped: only ever decremented)
    int32_t *core;
    uint32_t *layer;
    uint32_t *alive[2];
    uint64_t *slices;                           // first_entry << 12 | (length - 1), length <= kOSliceLen
    uint32_t slice_cap;
    uint32_t log_cap;                           // entries per log (the largest n_local)
    OnionCtl *ctl_local;
    OnionCtl *ctl_peer[kMaxRanks];
    uint32_t *log_local[kMaxRanks];             // this rank's copy of rank q's log (q == rank: the log itself)
    uint32_t *log_peer[kMaxRanks];              // rank p's copy of THIS rank's log (peer memory)
    ORankState *st;
};

struct OShared {
    uint32_t first[kOThreads];                  // the batch of lists a CTA walks: first entry ...
    uint32_t off[kOThreads + 1];                // ... and exclusive prefix of the lengths
    uint32_t scan[kOWarps + 1];
    uint32_t base[2];
    unsigned long long src_lo[kMaxRanks], src_cnt[kMaxRanks];
    uint32_t bcast;
};

// The lanes with found set took a degree from k + 1 to k: they log their unitig into layer lnext with coreness k.
// Called by whole warps; one atomic on the log length per warp.
__device__ __forceinline__ void log_found(const ORank &R, ORankState *st, bool found, uint32_t loc, int32_t k, uint32_t lnext) {
    const uint32_t m = __ballot_sync(kFullMask, found);
    if (m == 0) return;
    uint32_t pos = 0;
    if (lane_id() == 0) pos = atomicAdd(&st->log_cnt, (uint32_t)__popc(m));
    pos = __shfl_sync(kFullMask, pos, 0) + __popc(m & lanemask_lt());
    if (!found) return;
    R.core[loc] = k;
    R.layer[loc] = lnext;
    if (pos < R.log_cap) R.log_local[R.rank][pos] = R.v_lo + loc;
    else atomicCAS(&st->error, 0u, (uint32_t)kErrFull);
}

// one decrement per lane (loc = ~0u: none).  Degrees never go up: a unitig at or below k is already in a log and is
// not touched again; look = false decrements without looking first (one round trip less on a thin chain).
__device__ __forceinline__ void relax(const ORank &R, ORankState *st, const uint32_t (&u)[kOUnroll], bool look, int32_t k, uint32_t lnext) {
    int32_t d[kOUnroll];
#pragma unroll
    for (int t = 0; t < kOUnroll; ++t) d[t] = u[t] == ~0u ? INT32_MIN : (look ? __ldcg(&R.deg[u[t]]) : INT32_MAX);
#pragma unroll
    for (int t = 0; t < kOUnroll; ++t) d[t] = d[t] > k ? atomicSub(&R.deg[u[t]], 1) : INT32_MIN;
#pragma unroll
    for (int t = 0; t < kOUnroll; ++t) log_found(R, st, d[t] == k + 1, u[t], k, lnext);
}

// WALK of the ids [c0, c1) of the concatenated fresh parts of all logs (sh.src_*) by the CTAs cta, cta + step, ...
// in tiles of `tile` ids.  slice_long: lists longer than kOSliceLen go to the slice list instead (walked after a barrier).
__device__ __forceinline__ void walk_ids(const ORank &R, ORankState *st, OShared &sh, unsigned long long total_ids, uint32_t cta, uint32_t nctas,
                                         uint32_t tile, bool slice_long, int32_t k, uint32_t lnext) {
    const uint32_t tid = threadIdx.x;
    for (unsigned long long t0 = (unsigned long long)cta * tile; t0 < total_ids; t0 += (unsigned long long)nctas * tile) {
        const unsigned long long i = t0 + tid;
        uint32_t first = 0, len = 0;
        if (tid < tile && i < total_ids) {
            unsigned long long off = i;
            int q = 0;
            while (off >= sh.src_cnt[q]) { off -= sh.src_cnt[q]; ++q; }   // i < total_ids: q stays < world
            const uint32_t x = log_read(&R.log_local[q][sh.src_lo[q] + off], st);
            if (x >= R.n_global) {
                atomicCAS(&st->error, 0u, (uint32_t)kErrBadEntry);
            } else {
                first = R.nbr_ptr[x];
                len = R.nbr_ptr[x + 1] - first;
            }
            if (slice_long && len > kOSliceLen) {
                const uint32_t ns = (len + kOSliceLen - 1) / kOSliceLen;
                const uint32_t s0 = atomicAdd(&st->slice_cnt, ns);
                for (uint32_t s = 0; s < ns; ++s) {
                    const uint32_t l = min(kOSliceLen, len - s * kOSliceLen);
                    if (s0 + s < R.slice_cap) R.slices[s0 + s] = ((uint64_t)(first + s * kOSliceLen) << 12) | (uint64_t)(l - 1u);
                    else atomicCAS(&st->error, 0u, (uint32_t)kErrFull);
                }
                len = 0;
            }
        }
        uint32_t total = 0;
        const uint32_t ex = block_excl_scan_add<uint32_t, kOThreads>(len, sh.scan, &total);
        sh.off[tid] = ex;
        sh.first[tid] = first;
        if (tid == 0) sh.off[kOThreads] = total;
        __syncthreads();
        const bool look = total > (uint32_t)kOThreads;
        for (uint32_t b = 0; b < total; b += kOThreads * kOUnroll) {
            uint32_t u[kOUnroll];
#pragma unroll
            for (int t = 0; t < kOUnroll; ++t) {
                const uint32_t e = b + t * kOThreads + tid;
                u[t] = ~0u;
                if (e < total) {
                    uint32_t lo = 0, hi = kOThreads;   // off[lo] <= e < off[hi]: the last list that starts at or before e
#pragma unroll
                    for (int s = 0; s < 9; ++s) {
                        const uint32_t mid = (lo + hi) >> 1;
                        if (sh.off[mid] <= e) lo = mid; else hi = mid;
                    }
                    u[t] = R.nbr[sh.first[lo] + (e - sh.off[lo])];
                }
            }
            relax(R, st, u, look, k, lnext);
        }
        __syncthreads();   // off / first are reused by the next tile
    }
}

// the slices of this step's long lists, one per CTA at a time
__device__ __forceinline__ void walk_slices(const ORank &R, ORankState *st, uint32_t cta, uint32_t nctas, int32_t k, uint32_t lnext) {
    const uint32_t n_sl = min(__ldcg(&st->slice_cnt), R.slice_cap);
    for (uint32_t s = cta; s < n_sl; s += nctas) {
        const uint64_t sl = __ldcg(&R.slices[s]);
        const uint32_t first = (uint32_t)(sl >> 12), len = (uint32_t)(sl & 0xfffu) + 1u;
        for (uint32_t b = 0; b < len; b += kOThreads * kOUnroll) {
            uint32_t u[kOUnroll];
#pragma unroll
            for (int t = 0; t < kOUnroll; ++t) {
                const uint32_t e = b + t * kOThreads + threadIdx.x;
                u[t] = e < len ? R.nbr[first + e] : ~0u;
            }
            relax(R, st, u, true, k, lnext);
        }
    }
}

// SCAN of level k (all CTAs of the rank): alive unitigs at degree k are logged as layer lnum, survivors compacted
__device__ __forceinline__ void scan_level(const ORank &R, ORankState *st, uint32_t cta, const uint32_t *alive_src, uint32_t n_alive,
                                           uint32_t *alive_dst, uint32_t *alive_out, int32_t k, uint32_t lnum, OShared &sh) {
    const uint32_t tid = threadIdx.x;
    int32_t local_min = INT32_MAX;
    const uint32_t tile = kOThreads * kOScanItems;
    uint32_t *log = R.log_local[R.rank];
    for (uint64_t t0 = (uint64_t)cta * tile; t0 < n_alive; t0 += (uint64_t)R.ctas * tile) {
        uint32_t v[kOScanItems], flag[kOScanItems];   // 1 = logged, 0x10000 = survivor
        uint32_t mine = 0;
#pragma unroll
        for (int j = 0; j < kOScanItems; ++j) {
            const uint64_t i = t0 + (uint64_t)j * kOThreads + tid;
            flag[j] = 0;
            v[j] = 0;
            if (i < n_alive) {
                v[j] = alive_src ? __ldcg(&alive_src[i]) : (uint32_t)i;
                const int32_t d = __ldcg(&R.deg[v[j]]);
                if (d == k) {
                    R.core[v[j]] = k;
                    R.layer[v[j]] = lnum;
                    flag[j] = 1u;
                } else if (d > k) {
                    flag[j] = 0x10000u;
                    local_min = min(local_min, d);
                }
            }
            mine += flag[j];
        }
        uint32_t total = 0;
        const uint32_t ex = block_excl_scan_add<uint32_t, kOThreads>(mine, sh.scan, &total);
        if (tid == 0) {
            const uint32_t nf = total & 0xffffu, ns = total >> 16;
            sh.base[0] = nf ? atomicAdd(&st->log_cnt, nf) : 0;
            sh.base[1] = ns ? atomicAdd(alive_out, ns) : 0;
        }
        __syncthreads();
        uint32_t fpos = sh.base[0] + (ex & 0xffffu), spos = sh.base[1] + (ex >> 16);
#pragma unroll
        for (int j = 0; j < kOScanItems; ++j) {
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

// The meeting that ends step t, by the leader warp (CTA 0, warp 0); lane q + 1 talks to rank q.  copy_here: the new
// part of the own log is short (a solo step) and this warp copies it to the peers itself.  Releases the plan of step
// t + 1: its kind, its level and the number of the last non-empty layer.
__device__ __forceinline__ void meet(const ORank &R, ORankState *st, uint32_t t, bool walked, int32_t k, uint32_t lnum, bool copy_here,
                                     unsigned long long &peer_log_hi, uint32_t &published) {
    const uint32_t lane = lane_id();
    const int world = R.world;
    const int peer = (int)lane - 1;
    const bool has_peer = peer >= 0 && peer < world;
    const uint32_t par = t & 1u;
    const unsigned long long tag = (unsigned long long)t << kTagShift;
    unsigned long long log_len = 0;
    int32_t lmin = INT32_MAX;
    if (lane == 0) {
        log_len = __ldcg(&st->log_cnt);
        lmin = __ldcg(&st->local_min);
        st->published = (uint32_t)log_len;
        st->local_min = INT32_MAX;
        st->slice_cnt = 0;   // every CTA has walked the slices (rank barrier) or none were made (solo)
    }
    log_len = __shfl_sync(kFullMask, log_len, 0);
    lmin = __shfl_sync(kFullMask, lmin, 0);
    const uint32_t pub_lo = published;
    published = (uint32_t)log_len;
    if (copy_here && world > 1 && lane > 0) {
        const uint32_t *src = R.log_local[R.rank];
        for (uint32_t i = pub_lo + (lane - 1u); i < (uint32_t)log_len; i += 31u) {
            const uint32_t x = __ldcg(&src[i]);
            for (int p = 0; p < world; ++p)
                if (p != R.rank) R.log_peer[p][i] = x;
        }
    }
    if (has_peer) {
        OnionCtl *dst = R.ctl_peer[peer];
        st_relaxed_sys(&dst->w[par][R.rank][1], tag | (unsigned long long)(uint32_t)lmin);
        st_relaxed_sys(&dst->w[par][R.rank][0], tag | log_len);
    }
    unsigned long long w0 = 0, w1 = (unsigned long long)(uint32_t)INT32_MAX;
    bool failed = false;
    if (has_peer) {
        const OnionCtl *mine = R.ctl_local;
        const unsigned long long t_wait = pglobal_ns();
        uint32_t spins = 0;
        while (true) {
            w0 = ld_relaxed_sys(&mine->w[par][peer][0]);
            w1 = ld_relaxed_sys(&mine->w[par][peer][1]);
            if ((w0 >> kTagShift) == t && (w1 >> kTagShift) == t) break;
            if ((++spins & 1023u) == 0 && (*(volatile uint32_t *)&st->error || pglobal_ns() - t_wait > kPeelWatchdogNs)) { failed = true; break; }
        }
        w0 &= kValMask;
        w1 &= kValMask;
    }
    if (__ballot_sync(kFullMask, failed)) {
        if (lane == 0) {
            atomicCAS(&st->error, 0u, (uint32_t)kErrPeers);
            st_rel_gpu(&st->plan[t % kOPlanRing], ((unsigned long long)t << 8) | kPlanDone);
        }
        return;
    }
    const unsigned long long before = peer_log_hi;
    if (has_peer) peer_log_hi = w0;
    unsigned long long g_fresh = 0, g_total = 0;
    uint32_t g_min = (uint32_t)INT32_MAX;
    for (int q = 0; q < world; ++q) {
        const unsigned long long hi = __shfl_sync(kFullMask, w0, q + 1);
        const unsigned long long lo = __shfl_sync(kFullMask, before, q + 1);
        g_min = min(g_min, (uint32_t)__shfl_sync(kFullMask, w1, q + 1));
        g_total += hi;
        g_fresh += hi - lo;
        if (lane == 0) {
            st->log_lo[q] = lo;
            st->log_hi[q] = hi;
        }
    }
    // every lane derives the same plan
    uint32_t flags = kPlanFull;
    int32_t k_next = k;
    uint32_t l_next = lnum;
    if (g_fresh) {
        // a layer was formed: walk it next, unless it holds the last unitigs of the graph
        l_next = lnum + 1;
        flags = g_total >= R.n_global ? kPlanDone : kPlanWalk | kPlanFull;
    } else if (g_total >= R.n_global) {
        flags = kPlanDone;                    // every unitig of the graph is in a log
    } else if (walked) {
        k_next = k + 1;                       // the level is over
    } else if (g_min == (uint32_t)INT32_MAX) {
        flags = kPlanDone;                    // nothing alive anywhere (the host reports the unitigs not placed)
    } else {
        k_next = (int32_t)g_min;              // the level was empty: skip to the smallest surviving degree
    }
    if ((flags & kPlanWalk) && g_fresh <= kSoloIds) {
        // the local entries the walk would visit: few, and this rank runs the step on CTA 0 alone
        unsigned long long edges = 0;
        for (int q = 0; q < world; ++q) {
            const unsigned long long hi = __shfl_sync(kFullMask, w0, q + 1), lo = __shfl_sync(kFullMask, before, q + 1);
            for (unsigned long long i = lo + lane; i < hi; i += 32u) {
                const uint32_t x = log_read(&R.log_local[q][i], st);
                if (x < R.n_global) edges += R.nbr_ptr[x + 1] - R.nbr_ptr[x];
            }
        }
        for (int s = 16; s > 0; s >>= 1) edges += __shfl_xor_sync(kFullMask, edges, s);
        if (edges <= kSoloEdges) flags &= ~kPlanFull;
    }
    if (lane == 0) {
        st->meetings = t;
        if (g_fresh && !walked) st->levels += 1;
        if (!(flags & kPlanFull)) st->solo_steps += 1;
        st->n_layers = l_next;
        st->plan_k[t % kOPlanRing] = k_next;
        st->plan_layer[t % kOPlanRing] = l_next;
        st_rel_gpu(&st->plan[t % kOPlanRing], ((unsigned long long)t << 8) | flags);
    }
}

__global__ void __launch_bounds__(kOThreads, 2) ponion_kernel(const ORank *ranks, uint32_t ctas_per_rank) {
    __shared__ OShared sh;
    const ORank &R = ranks[blockIdx.x / ctas_per_rank];   // read in place: a copy would live in local memory
    ORankState *st = R.st;
    const uint32_t cta = blockIdx.x % ctas_per_rank;
    const uint32_t tid = threadIdx.x, warp = tid >> 5;
    const bool leader_cta = cta == 0;
    unsigned long long bar_gen = 0;
    uint32_t t = 1;                          // step number (tags of zero-initialised control words are 0)
    uint32_t flags = kPlanFull;              // step 1: the scan of level 0
    int32_t k = 0;
    uint32_t lnum = 0;                       // the number of the last non-empty layer
    const uint32_t *alive_src = nullptr;     // nullptr: every local unitig
    uint32_t alive_i = 0, n_alive = R.n_local;
    unsigned long long peer_log_hi = 0;      // leader warp, lane q + 1: length of rank q's log at the last meeting
    uint32_t published = 0;                  // leader warp: length of the own log at the last meeting

    while (!(flags & kPlanDone)) {
        const bool walk = flags & kPlanWalk, full = flags & kPlanFull;
        if ((t % kOPlanSync) == 0) rank_barrier(st, R.ctas, bar_gen, false);   // bounds CTA 0's lead (plan ring)
        if (walk && (full || leader_cta)) {
            if (tid < kMaxRanks) {
                unsigned long long lo = 0, cnt = 0;
                if ((int)tid < R.world) {
                    lo = __ldcg(&st->log_lo[tid]);
                    cnt = __ldcg(&st->log_hi[tid]) - lo;
                }
                sh.src_lo[tid] = lo;
                sh.src_cnt[tid] = cnt;
            }
            __syncthreads();
            unsigned long long total = 0;
            for (int q = 0; q < R.world; ++q) total += sh.src_cnt[q];
            if (full) {
                const uint32_t tile = (uint32_t)min((unsigned long long)kOThreads, max(1ull, (total + R.ctas - 1) / R.ctas));
                walk_ids(R, st, sh, total, cta, R.ctas, tile, true, k, lnum + 1);
                rank_barrier(st, R.ctas, bar_gen, false);   // every slice of the step is listed
                walk_slices(R, st, cta, R.ctas, k, lnum + 1);
                rank_barrier(st, R.ctas, bar_gen, false);
            } else {
                walk_ids(R, st, sh, total, 0, 1, kOThreads, false, k, lnum + 1);
                __syncthreads();
                if (tid == 0) __threadfence();
                __syncthreads();
            }
        } else if (!walk) {
            scan_level(R, st, cta, alive_src, n_alive, R.alive[alive_i], &st->alive_out[alive_i], k, lnum + 1, sh);
            rank_barrier(st, R.ctas, bar_gen, false);
            n_alive = __ldcg(&st->alive_out[alive_i]);
            alive_src = R.alive[alive_i];
            alive_i ^= 1u;
            // the other slot was last read two scans ago (every CTA has passed a barrier since): re-arm it
            if (leader_cta && tid == 0) st->alive_out[alive_i] = 0;
        }
        // publish: on all CTAs when they all worked; a solo step's few ids are copied by the leader warp as it meets
        if (full && R.world > 1) {
            publish_stage(R, st, cta * kOThreads + tid, R.ctas * kOThreads);
            rank_barrier(st, R.ctas, bar_gen, false);
        }
        if (leader_cta && warp == 0) meet(R, st, t, walk, k, lnum, !full, peer_log_hi, published);
        flags = wait_plan<kPlanDone>(&st->plan[t % kOPlanRing], t, st, &sh.bcast);
        k = __ldcg(&st->plan_k[t % kOPlanRing]);
        lnum = __ldcg(&st->plan_layer[t % kOPlanRing]);
        if (*(volatile uint32_t *)&st->error) break;
        ++t;
        if (t >= (1u << 24) - 2u) { if (tid == 0) atomicCAS(&st->error, 0u, (uint32_t)kErrBarrier); break; }
    }
}

}  // namespace

int dist_onion(kombgpu_dist_graph *g) {
    kombgpu_comm *c = g->comm;
    kombgpu_ctx *ctx = g->ctx;
    const int world = c->world;
    const uint32_t n_local = g->n_local;
    dist_onion_release(g);
    DistOnionInfo info{};

    // everything a rank needs before the kernel; a rank that fails here still meets the others below, and every
    // rank returns an error there: nobody is left waiting on the device
    DevBuf<uint32_t> t_ptr, t_nbr, layer, alive_a, alive_b;
    DevBuf<int32_t> core, work;
    DevBuf<uint64_t> slices;
    DevBuf<ORankState> state;
    DevBuf<ORank> desc;
    const uint32_t log_cap = g->step;   // the largest n_local
    SymRewind heap{c, sym_mark(c)};   // the logs and control words, given back on every return path
    uint32_t *logs = nullptr;
    PeerPtrs<uint32_t> logs_peers{};
    OnionCtl *ctl = nullptr;
    PeerPtrs<OnionCtl> ctl_peers{};
    // every unitig of the graph is walked once on each rank: sum of ceil(len / kOSliceLen) over the long lists
    const uint64_t slice_cap64 = 2 * g->n_directed / kOSliceLen + 1;
    uint32_t ctas_per_rank = 0;
    ORank R{};
    int rc = sym_alloc(c, (size_t)world * log_cap, &logs, &logs_peers);
    rc = first_rc(rc, sym_alloc(c, 1, &ctl, &ctl_peers));
    if (rc == KOMBGPU_OK) rc = [&]() -> int {
        const uint32_t *nbr_ptr = g->nbr_ptr, *nbr = g->nbr;
        if (!nbr_ptr) {
            // the build laid out rows for the asynchronous or replicated peel: the onion walks their transpose
            EvTimer tt(ctx);
            KG_TRY(dist_rows_to_nbr(g, t_ptr, t_nbr));
            info.ms_transpose = tt.lap();
            nbr_ptr = t_ptr.p;
            nbr = t_nbr.p;
        }
        if (slice_cap64 >= 0xffffffffull) return ctx_fail(ctx, KOMBGPU_EINVAL, "partition too large for the onion's slice list");
        KG_CUDA(ctx, cudaMemsetAsync(ctl, 0, sizeof(OnionCtl), ctx->stream));
        KG_CUDA(ctx, cudaMemsetAsync(logs, 0xff, (size_t)world * log_cap * sizeof(uint32_t), ctx->stream));   // kLogEmpty
        KG_ALLOC(ctx, layer, n_local);
        KG_ALLOC(ctx, core, n_local);
        KG_ALLOC(ctx, work, n_local);
        KG_ALLOC(ctx, alive_a, n_local);
        KG_ALLOC(ctx, alive_b, n_local);
        KG_ALLOC(ctx, slices, slice_cap64);
        KG_ALLOC(ctx, state, 1);
        KG_ALLOC(ctx, desc, kMaxRanks);
        KG_CUDA(ctx, cudaMemsetAsync(layer.p, 0, (size_t)(n_local ? n_local : 1) * sizeof(uint32_t), ctx->stream));
        KG_CUDA(ctx, cudaMemsetAsync(core.p, 0, (size_t)(n_local ? n_local : 1) * sizeof(int32_t), ctx->stream));
        if (n_local) KG_CUDA(ctx, cudaMemcpyAsync(work.p, g->deg, (size_t)n_local * sizeof(int32_t), cudaMemcpyDeviceToDevice, ctx->stream));
        ORankState init{};
        init.local_min = INT32_MAX;
        KG_CUDA(ctx, cudaMemcpyAsync(state.p, &init, sizeof(init), cudaMemcpyHostToDevice, ctx->stream));
        KG_TRY(rank_ctas(ctx, c, ponion_kernel, kOThreads, 1, &ctas_per_rank));
        R.n_local = n_local; R.v_lo = g->v_lo; R.n_global = g->n_global; R.world = world; R.rank = c->rank; R.ctas = ctas_per_rank;
        R.nbr_ptr = nbr_ptr; R.nbr = nbr; R.deg = work.p; R.core = core.p; R.layer = layer.p;
        R.alive[0] = alive_a.p; R.alive[1] = alive_b.p;
        R.slices = slices.p; R.slice_cap = (uint32_t)slice_cap64;
        R.log_cap = log_cap;
        R.ctl_local = ctl;
        for (int q = 0; q < world; ++q) {
            R.ctl_peer[q] = ctl_peers.p[q];
            R.log_local[q] = logs + (size_t)q * log_cap;                         // my copy of rank q's log
            R.log_peer[q] = logs_peers.p[q] + (size_t)c->rank * log_cap;        // rank q's copy of my log
        }
        R.st = state.p;
        KG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));   // the control words are cleared before any peer publishes
        return KOMBGPU_OK;
    }();
    KG_TRY(barrier_rc(c, rc));

    const cudaError_t le = launch_ranks(c, ponion_kernel, kOThreads, ctas_per_rank, R, desc.p, &info.ms_kernel);
    if (le != cudaSuccess) rc = ctx_fail(ctx, KOMBGPU_ECUDA, "partitioned onion kernel: %s", cudaGetErrorString(le));
    ORankState fin{};
    if (rc == KOMBGPU_OK) rc = read_back(ctx, state.p, &fin, 1);
    // global figures; also: nobody gives back its logs (at return) while a peer may still be writing
    uint32_t ms_bits = 0;
    memcpy(&ms_bits, &info.ms_kernel, sizeof(ms_bits));
    unsigned long long mine[5] = {fin.error, fin.log_cnt, fin.n_layers, fin.meetings, ms_bits}, all[kMaxRanks * 5];
    KG_TRY(exchange_rc(c, rc, mine, 5, all));
    if (c->same_device) {
        // every rank ran inside rank 0's launch, which its events timed
        ms_bits = (uint32_t)all[4];
        memcpy(&info.ms_kernel, &ms_bits, sizeof(ms_bits));
    }
    uint64_t placed = 0;
    for (int q = 0; q < world; ++q) {
        if (all[q * 5]) return ctx_fail(ctx, KOMBGPU_EINTERNAL, "partitioned onion: rank %d reports error %llu (%s)", q, all[q * 5], rank_error_text(all[q * 5]));
        placed += all[q * 5 + 1];
        if (all[q * 5 + 2] != fin.n_layers || all[q * 5 + 3] != fin.meetings)
            return ctx_fail(ctx, KOMBGPU_EINTERNAL, "partitioned onion: rank %d ended at layer %llu after %llu meetings, rank %d at %u after %u", q,
                            all[q * 5 + 2], all[q * 5 + 3], c->rank, fin.n_layers, fin.meetings);
    }
    if (placed != g->n_global) return ctx_fail(ctx, KOMBGPU_EINTERNAL, "partitioned onion ended with %llu of %u unitigs placed", (unsigned long long)placed, g->n_global);
    info.levels = fin.levels;
    info.meetings = fin.meetings;
    info.solo_steps = fin.solo_steps;
    g->onion_layer = layer.take();
    g->onion_core = core.take();
    g->onion_n_layers = fin.n_layers;
    g->onion_info = info;
    g->has_onion = true;
    if (getenv("KOMBGPU_DEBUG"))
        fprintf(stderr, "[kombgpu] rank %d ponion: layers %u levels %u meetings %u solo %u ctas %u kernel %.3f ms transpose %.3f ms\n", c->rank,
                fin.n_layers, fin.levels, fin.meetings, fin.solo_steps, ctas_per_rank, info.ms_kernel, info.ms_transpose);
    return KOMBGPU_OK;
}

void dist_onion_release(kombgpu_dist_graph *g) {
    if (g->onion_layer) ws_free(g->ctx, g->onion_layer);
    if (g->onion_core) ws_free(g->ctx, g->onion_core);
    g->onion_layer = nullptr;
    g->onion_core = nullptr;
    g->onion_n_layers = 0;
    g->has_onion = false;
}

}  // namespace kg

using namespace kg;

extern "C" {

int kombgpu_dist_onion(kombgpu_dist_graph *g, uint32_t *layer, uint32_t *n_layers) {
    if (!g) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = g->ctx;
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    if (!g->has_onion) KG_TRY(dist_onion(g));
    if (n_layers) *n_layers = g->onion_n_layers;
    if (layer && g->n_local) {
        KG_CUDA(ctx, cudaMemcpyAsync(layer, g->onion_layer, (size_t)g->n_local * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
        KG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return KOMBGPU_OK;
}

// measurement aids (include/kombgpu_debug.h)
int kombgpu_debug_dist_onion_again(kombgpu_dist_graph *g) {
    if (!g) return KOMBGPU_EINVAL;
    g->has_onion = false;
    return kombgpu_dist_onion(g, nullptr, nullptr);
}

int kombgpu_debug_dist_onion_timing(const kombgpu_dist_graph *g, float *ms_kernel, uint32_t *levels, uint32_t *meetings, uint32_t *solo_steps,
                                    float *ms_transpose) {
    if (!g) return KOMBGPU_EINVAL;
    if (!g->has_onion) return ctx_fail(g->ctx, KOMBGPU_ESTATE, "kombgpu_dist_onion has not run");
    if (ms_kernel) *ms_kernel = g->onion_info.ms_kernel;
    if (levels) *levels = g->onion_info.levels;
    if (meetings) *meetings = g->onion_info.meetings;
    if (solo_steps) *solo_steps = g->onion_info.solo_steps;
    if (ms_transpose) *ms_transpose = g->onion_info.ms_transpose;
    return KOMBGPU_OK;
}

}  // extern "C"
