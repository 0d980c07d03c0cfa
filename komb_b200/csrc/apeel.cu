// apeel.cu — stage 2 over the ranks of a communicator, ASYNCHRONOUS form: the k-core peel of a graph partitioned by
// unitig-id range with no meeting of the ranks inside a level.
//
// Replaces igraph_coreness (src/graph.cpp:463) like peel.cu (one GPU) and ppeel.cu (ranks that meet once per
// cascade generation); the result is the same unique function of the graph, bit-exact whatever the partition.
//
// One persistent kernel per GPU.  A rank owns the rows, the working degrees and the POOL of its own unitigs; degrees
// and pools live in the symmetric heap, so every rank can reach every other rank's over NVLink.
//   worker warps   hold a ticket of their rank's pool and spin on that slot alone (slots are written once and valid
//                  when they differ from an EMPTY marker).  The warp that receives unitig v at level k stores
//                  core[v] = k, walks v's row and decrements every neighbour where it lives -- atom.sys on the owner's
//                  degree slice, local or remote.  Degrees are never clamped and only go down, so the decrement that
//                  takes a degree from k + 1 to k owns that unitig: the same lane fetch-adds the OWNER's pool tail
//                  and stores (k, id) into the slot it got.  Whoever holds that ticket wakes up.  Rows longer than
//                  kASlice entries are cut into slices that go through the owner's own pool.
//   manager warp   (CTA 0) drives the levels: [min] the smallest surviving degree on this rank -> exchanged through
//                  tagged words in peer memory -> the next level k; [scan] unitigs at degree k are pushed, survivors
//                  compacted; a flag exchange makes sure every rank's scan is complete before anybody decrements;
//                  then workers are released and the manager watches for the end of the level.
//   end of level   every rank counts entries pushed into its pool (tail: bumped by the PRODUCER before its own entry
//                  counts as done) and entries processed (done).  All ranks idle at one instant <=> the level is over;
//                  a manager reads done then tail of every rank, and the tails once more: equal and unchanged means
//                  such an instant existed (a rank cannot receive work while everybody's done == tail).
// Inside a level nothing waits for anything but its own ticket: a cascade step costs one remote atomic, one remote
// fetch-add and one remote store, not a meeting of all ranks.
//
// Ranks that share one device (tests) run inside ONE grid, a group of CTAs per rank.
#include <cstdio>
#include <cstdlib>

#include "prank.cuh"

namespace kg {
namespace {

constexpr int kAThreads = 512;
constexpr int kAWarps = kAThreads / 32;
constexpr int kAU = 4;                        // independent decrement chains per lane
constexpr uint32_t kASlice = 256;             // rows longer than this are cut into slices of this many entries (a slice is walked by one warp,
                                              // 128 entries per round trip: cfg5 on 2 GPUs took 7.7 s with 2048-entry slices)
constexpr int kAScanItems = 8;
constexpr unsigned long long kAEmpty = ~0ull;
constexpr unsigned long long kASliceFlag = 1ull << 63;   // entry = flag | piece << 32 | local id ; else k << 32 | local id
constexpr int kALvlProf = 48;

enum : uint32_t { kPhMin = 1, kPhScan = 2, kPhGo = 3, kPhExit = 4 };

// symmetric control block, one per rank
struct ACtl {
    unsigned long long q_tail;                 // entries pushed into this rank's pool (fetch-add by any rank)
    unsigned long long pad0[15];
    unsigned long long q_done;                 // entries this rank has processed
    unsigned long long pad1[15];
    unsigned long long min_next[kMaxRanks];    // written by rank src: epoch << 32 | its smallest surviving degree
    unsigned long long scan_seen[kMaxRanks];   // written by rank src: epoch of its last completed scan
};

struct AState {   // local to a rank
    unsigned long long q_head;                 // tickets handed out
    unsigned long long phase_word;             // seq << 40 | type << 32 | level (of a SCAN / GO)
    unsigned long long phase_done;             // worker CTAs that finished a phase (cumulative)
    unsigned long long n_visited, n_remote_dec, n_remote_push, n_slices, n_own_push;   // own: pushed into the own pool (scan, local discoveries, slices)
    unsigned long long prof_ns[6];             // manager: 0 min pass, 1 min exchange, 2 scan pass, 3 scan exchange, 4 level (go -> over)
    uint32_t alive_cnt[2];
    uint32_t n_alive, alive_src;               // parameters of the current phase: list length, list index (2 = identity)
    int32_t local_min, cur_k, prev_k, max_core;
    uint32_t levels, error;                    // error: kErr*
    uint32_t lvl_ns[kALvlProf], lvl_pushed[kALvlProf];   // first levels: time from GO to the end of the level, entries this rank processed
    int32_t lvl_k[kALvlProf];
};

struct ARank {
    uint32_t n_local, v_lo, n_global, step;
    int world, rank;
    uint32_t ctas;                             // CTAs of this rank: CTA 0 manages, the rest work
    const uint32_t *row_ptr;                   // [n_local + 1]
    const uint32_t *col;                       // global neighbour ids
    int32_t *core;
    uint32_t *alive[2];
    uint32_t pool_cap;
    int32_t *deg_peer[kMaxRanks];
    unsigned long long *pool_peer[kMaxRanks];
    ACtl *ctl_peer[kMaxRanks];
    uint8_t *dead_peer[kMaxRanks];             // every rank's map of peeled unitigs (global ids): written by the owners, read locally
    AState *st;
};

// ---- worker side ------------------------------------------------------------------------------------------------

// decrement the neighbours col[lo, hi) of a unitig peeled at level k (whole warp)
__device__ __forceinline__ void a_walk(const ARank &R, AState *st, uint32_t lo, uint32_t hi, int32_t k, bool use_map) {
    const uint32_t lane = lane_id();
    unsigned long long n_remote = 0, n_push = 0, n_own = 0;
    int32_t left = INT32_MAX;   // smallest degree above k this walk left behind
    const uint8_t *dead = use_map ? R.dead_peer[R.rank] : nullptr;
    for (uint32_t base = lo; base < hi; base += 32u * kAU) {
        uint32_t own[kAU], li[kAU];
        int32_t old[kAU];
#pragma unroll
        for (int t = 0; t < kAU; ++t) {
            const uint32_t e = base + t * 32u + lane;
            own[t] = 0xffffffffu;
            if (e < hi) {
                const uint32_t u = R.col[e];
                // a unitig already peeled needs no decrement: its owner marked it in every rank's map when it peeled it (the
                // mark may still be on its way: then the decrement is merely wasted)
                if (!dead || !__ldcg(&dead[u])) {
                    own[t] = u / R.step;
                    li[t] = u - own[t] * R.step;
                }
            }
        }
#pragma unroll
        for (int t = 0; t < kAU; ++t) {
            old[t] = INT32_MIN;
            if (own[t] != 0xffffffffu) {
                old[t] = atomicSub_system(R.deg_peer[own[t]] + li[t], 1);
                n_remote += own[t] != (uint32_t)R.rank;
            }
        }
#pragma unroll
        for (int t = 0; t < kAU; ++t)
            if (old[t] > k + 1) left = min(left, old[t] - 1);
#pragma unroll
        for (int t = 0; t < kAU; ++t) {
            if (old[t] == k + 1) {   // this decrement took the unitig to level k: it is peeled now, by its owner
                const unsigned long long tk = atomicAdd_system(&R.ctl_peer[own[t]]->q_tail, 1ull);
                if (tk < R.pool_cap) st_relaxed_sys(R.pool_peer[own[t]] + tk, ((unsigned long long)(uint32_t)k << 32) | li[t]);
                else atomicCAS(&st->error, 0u, (uint32_t)kErrFull);
                n_push += own[t] != (uint32_t)R.rank;
                n_own += own[t] == (uint32_t)R.rank;
            }
        }
    }
    n_remote = warp_reduce_add(n_remote);
    n_push = warp_reduce_add(n_push);
    n_own = warp_reduce_add(n_own);
    left = warp_reduce_min(left);
    __syncwarp();
    if (lane == 0) {
        atomicAdd(&st->n_visited, (unsigned long long)(hi - lo));
        if (n_remote) atomicAdd(&st->n_remote_dec, n_remote);
        if (n_push) atomicAdd(&st->n_remote_push, n_push);
        if (n_own) atomicAdd(&st->n_own_push, n_own);
        // the bound must be in place before this entry counts as done (the manager reads it after the level's end): a
        // RETURNING atomic has been performed when its value arrives, and the increment below is made to depend on that
        // value -- no fence (a membar here was 11 % of the kernel's stall samples)
        unsigned long long one = 1ull;
        if (left != INT32_MAX) one += (unsigned long long)(atomicMin(&st->local_min, left) == INT32_MIN);   // never true: degrees are >= 0
        // every decrement of this entry has returned and every unitig it discovered is counted in its owner's tail
        atomicAdd_system(&R.ctl_peer[R.rank]->q_done, one);
    }
}

// The map of peeled unitigs saves the decrements of neighbours that are gone (half of all decrements), but looking a
// neighbour up before decrementing it adds a load to a cascade's critical path.  So it is consulted only while the pool
// holds a backlog (the level is bound by the rate of decrements, not by the length of a chain): measured on 8 GPUs with
// cfg2 x 8, always on: the last level 4.9 -> 3.1 ms, the level before it (277 dependent generations) 3.6 -> 4.0 ms.
constexpr unsigned long long kABacklog = 4096;

__device__ __forceinline__ void a_process(const ARank &R, AState *st, unsigned long long entry, unsigned long long ticket) {
    const uint32_t lane = lane_id();
    const bool use_map = R.dead_peer[R.rank] != nullptr &&
                         *(volatile unsigned long long *)&R.ctl_peer[R.rank]->q_tail > ticket + kABacklog;
    const uint32_t v = (uint32_t)entry;
    if (v >= R.n_local) { atomicCAS(&st->error, 0u, (uint32_t)kErrBadEntry); return; }
    const uint32_t row_lo = R.row_ptr[v], row_hi = R.row_ptr[v + 1];
    if (entry & kASliceFlag) {
        const uint32_t piece = (uint32_t)(entry >> 32) & 0x1fffffu;
        const int32_t k = *(volatile int32_t *)&st->cur_k;   // slices are made and walked inside one level, on this rank
        const uint32_t lo = row_lo + piece * kASlice;
        a_walk(R, st, lo, min(lo + kASlice, row_hi), k, use_map);
        return;
    }
    const int32_t k = (int32_t)((entry >> 32) & 0x7fffffffu);
    if (lane == 0) R.core[v] = k;
    if ((int)lane < R.world && R.dead_peer[lane]) R.dead_peer[lane][R.v_lo + v] = 1;   // lane q tells rank q
    uint32_t hi = row_hi;
    const uint32_t len = row_hi - row_lo;
    if (len > kASlice) {
        const uint32_t n_extra = (len - 1u) / kASlice;   // pieces 1 .. n_extra go through the pool, piece 0 is walked here
        unsigned long long pos = 0;
        if (lane == 0) {
            pos = atomicAdd_system(&R.ctl_peer[R.rank]->q_tail, (unsigned long long)n_extra);
            atomicAdd(&st->n_slices, (unsigned long long)n_extra);
            atomicAdd(&st->n_own_push, (unsigned long long)n_extra);
        }
        pos = __shfl_sync(kFullMask, pos, 0);
        for (uint32_t j = lane; j < n_extra; j += 32u) {
            if (pos + j < R.pool_cap) st_relaxed_sys(R.pool_peer[R.rank] + pos + j, kASliceFlag | ((unsigned long long)(j + 1u) << 32) | v);
            else atomicCAS(&st->error, 0u, (uint32_t)kErrFull);
        }
        hi = row_lo + kASlice;
    }
    a_walk(R, st, row_lo, hi, k, use_map);
}

// MIN phase (all threads of a worker CTA): the smallest degree above prev_k among the listed unitigs
__device__ __forceinline__ void a_phase_min(const ARank &R, AState *st, uint32_t wcta, uint32_t n_wctas) {
    const uint32_t n = st->n_alive, src = st->alive_src;
    const int32_t prev_k = st->prev_k;
    const int32_t *deg = R.deg_peer[R.rank];
    int32_t m = INT32_MAX;
    for (uint64_t i = (uint64_t)wcta * kAThreads + threadIdx.x; i < n; i += (uint64_t)n_wctas * kAThreads) {
        const uint32_t v = src < 2u ? __ldcg(&R.alive[src][i]) : (uint32_t)i;
        const int32_t d = __ldcg(&deg[v]);
        if (d > prev_k) m = min(m, d);
    }
    m = warp_reduce_min(m);
    if (lane_id() == 0 && m != INT32_MAX) atomicMin(&st->local_min, m);
}

// SCAN phase of level k: listed unitigs at degree k are pushed into the own pool, those above it are kept
__device__ __forceinline__ void a_phase_scan(const ARank &R, AState *st, uint32_t wcta, uint32_t n_wctas, uint32_t *s_scan, uint32_t *s_base,
                                             unsigned long long *s_base64) {
    const uint32_t n = st->n_alive, src = st->alive_src, dst = src == 0u ? 1u : 0u;
    const int32_t k = st->cur_k;
    const int32_t *deg = R.deg_peer[R.rank];
    const uint32_t tid = threadIdx.x;
    const uint32_t tile = kAThreads * kAScanItems;
    unsigned long long *pool = R.pool_peer[R.rank];
    int32_t surv_min = INT32_MAX;
    for (uint64_t t0 = (uint64_t)wcta * tile; t0 < n; t0 += (uint64_t)n_wctas * tile) {
        uint32_t v[kAScanItems], flag[kAScanItems], mine = 0;
        int32_t d[kAScanItems];
#pragma unroll
        for (int j = 0; j < kAScanItems; ++j) {   // ids first, then every degree: two round trips per tile, not two per item
            const uint64_t i = t0 + (uint64_t)j * kAThreads + tid;
            v[j] = i < n ? (src < 2u ? __ldcg(&R.alive[src][i]) : (uint32_t)i) : 0xffffffffu;
        }
#pragma unroll
        for (int j = 0; j < kAScanItems; ++j) d[j] = v[j] != 0xffffffffu ? __ldcg(&deg[v[j]]) : INT32_MIN;
#pragma unroll
        for (int j = 0; j < kAScanItems; ++j) {
            flag[j] = d[j] == k ? 1u : (d[j] > k ? 0x10000u : 0u);
            if (d[j] > k) surv_min = min(surv_min, d[j]);
            mine += flag[j];
        }
        uint32_t total = 0;
        const uint32_t ex = block_excl_scan_add<uint32_t, kAThreads>(mine, s_scan, &total);
        if (tid == 0) {
            const uint32_t nf = total & 0xffffu, ns = total >> 16;
            *s_base64 = nf ? atomicAdd_system(&R.ctl_peer[R.rank]->q_tail, (unsigned long long)nf) : 0ull;
            if (nf) atomicAdd(&st->n_own_push, (unsigned long long)nf);
            s_base[0] = ns ? atomicAdd(&st->alive_cnt[dst], ns) : 0u;
        }
        __syncthreads();
        unsigned long long fpos = *s_base64 + (ex & 0xffffu);
        uint32_t spos = s_base[0] + (ex >> 16);
#pragma unroll
        for (int j = 0; j < kAScanItems; ++j) {
            if (flag[j] == 1u) {
                if (fpos < R.pool_cap) st_relaxed_sys(pool + fpos, ((unsigned long long)(uint32_t)k << 32) | v[j]);
                else atomicCAS(&st->error, 0u, (uint32_t)kErrFull);
                ++fpos;
            } else if (flag[j]) {
                R.alive[dst][spos++] = v[j];
            }
        }
        __syncthreads();
    }
    surv_min = warp_reduce_min(surv_min);
    if (lane_id() == 0 && surv_min != INT32_MAX) atomicMin(&st->local_min, surv_min);
}

__device__ void a_worker(const ARank &R, uint32_t wcta, uint32_t n_wctas, uint32_t *s_scan, uint32_t *s_base, unsigned long long *s_base64) {
    AState *st = R.st;
    const uint32_t lane = lane_id();
    unsigned long long seen = 0;    // sequence number of the last phase word handled
    int32_t go_k = -1;              // the level this warp has seen released (GO): unitigs of that level may be peeled.  A scan
                                    // pushes its level's first unitigs BEFORE every rank's scan is complete; a warp that still
                                    // holds the previous level's release must not touch them (a decrement next to a scan in
                                    // progress peels a unitig twice).
    bool armed = false;             // between a GO and the next scan
    const unsigned long long *pool = R.pool_peer[R.rank];
    while (true) {
        unsigned long long t = 0;
        if (lane == 0) t = atomicAdd(&st->q_head, 1ull);
        t = __shfl_sync(kFullMask, t, 0);
        unsigned long long entry = kAEmpty;
        unsigned long long t0 = pglobal_ns();
        uint32_t spins = 0;
        while (true) {
            if (armed && t < R.pool_cap) {
                entry = ld_relaxed_sys(pool + t);
                // a slice only exists once its unitig's level was released; a unitig carries its level
                if (entry != kAEmpty && ((entry & kASliceFlag) || (int32_t)((entry >> 32) & 0x7fffffffu) == go_k)) break;
            }
            unsigned long long pw = *(volatile unsigned long long *)&st->phase_word;
            if ((pw >> 40) != seen) {
                pw = ld_acq_gpu(&st->phase_word);   // the phase's parameters were written before the word
                const uint32_t type = (uint32_t)(pw >> 32) & 0xffu;
                if (type == kPhExit) return;
                if (type == kPhGo) {
                    armed = true;
                    go_k = (int32_t)(uint32_t)pw;
                } else {
                    // MIN / SCAN are run by the whole CTA: every warp of it is in this loop (phases start when nothing is in flight)
                    armed = false;
                    __syncthreads();
                    if (type == kPhMin) a_phase_min(R, st, wcta, n_wctas);
                    else a_phase_scan(R, st, wcta, n_wctas, s_scan, s_base, s_base64);
                    __syncthreads();
                    if (threadIdx.x == 0) {
                        __threadfence();
                        atomicAdd(&st->phase_done, 1ull);
                    }
                }
                seen = pw >> 40;
                t0 = pglobal_ns();   // the peel is moving: the watchdog measures silence, not the length of the peel
                continue;
            }
            if ((++spins & 1023u) == 0) {
                if (*(volatile uint32_t *)&st->error) return;
                if (pglobal_ns() - t0 > kPeelWatchdogNs) { atomicCAS(&st->error, 0u, (uint32_t)kErrBarrier); return; }
            }
        }
        a_process(R, st, entry, t);
    }
}

// ---- manager side (one warp; lane q talks to rank q) ---------------------------------------------------------------

__device__ __forceinline__ bool a_issue_and_wait(const ARank &R, AState *st, unsigned long long &seq, uint32_t type, int32_t k,
                                                 unsigned long long &phases_run, bool wait) {
    ++seq;
    if (lane_id() == 0) st_rel_gpu(&st->phase_word, (seq << 40) | ((unsigned long long)type << 32) | (unsigned long long)(uint32_t)k);
    if (!wait) return true;
    ++phases_run;
    const unsigned long long want = phases_run * (unsigned long long)(R.ctas - 1u);
    bool ok = true;
    if (lane_id() == 0) {
        const unsigned long long t0 = pglobal_ns();
        uint32_t spins = 0;
        while (ld_acq_gpu(&st->phase_done) < want) {
            if ((++spins & 1023u) == 0 && (*(volatile uint32_t *)&st->error || pglobal_ns() - t0 > kPeelWatchdogNs)) { ok = false; break; }
        }
    }
    return __shfl_sync(kFullMask, ok ? 1 : 0, 0) != 0;
}

__device__ void a_manager(const ARank &R) {
    AState *st = R.st;
    const uint32_t lane = lane_id();
    const int world = R.world;
    const bool has_peer = (int)lane < world;
    ACtl *mine = R.ctl_peer[R.rank];
    unsigned long long seq = 0, phases_run = 0, epoch = 0;
    int32_t prev_k = -1;
    bool level_active = false;                // this rank processed entries in the level that just ended
    uint32_t n_alive = R.n_local, src = 2u;   // 2: every local unitig
    unsigned long long tp = pglobal_ns();
#define KG_APROF(slot)                                \
    if (lane == 0) {                                  \
        const unsigned long long now_ = pglobal_ns();       \
        st->prof_ns[slot] += now_ - tp;               \
        tp = now_;                                    \
    }
    bool failed = false;
    while (!failed) {
        // ---- a lower bound of the next level on this rank: the survivors' degrees as the last scan saw them and every
        //      degree a decrement of this rank left above the level (a unitig that died since only makes the bound lower:
        //      the level it names is then empty, which costs a scan, never a wrong answer).  Before the first level: a pass.
        if (epoch == 0) {
            if (lane == 0) {
                st->local_min = INT32_MAX;
                st->n_alive = n_alive;
                st->alive_src = src;
                st->prev_k = prev_k;
            }
            __syncwarp();
            if (!a_issue_and_wait(R, st, seq, kPhMin, -1, phases_run, true)) { failed = true; break; }
        }
        KG_APROF(0);
        ++epoch;
        int32_t lmin = 0;
        if (lane == 0) {
            lmin = *(volatile int32_t *)&st->local_min;
            st->local_min = INT32_MAX;   // the coming scan and level collect the next bound
        }
        lmin = __shfl_sync(kFullMask, lmin, 0);
        // bit 31: this rank peeled something in the level that just ended (a level named by a stale bound can be empty everywhere)
        const unsigned long long active_bit = level_active ? 0x80000000ull : 0ull;
        if (has_peer) st_relaxed_sys(&R.ctl_peer[lane]->min_next[R.rank], (epoch << 32) | active_bit | (unsigned long long)(uint32_t)lmin);
        int32_t gmin = INT32_MAX;
        bool any_active = false;
        {
            const unsigned long long t0 = pglobal_ns();
            uint32_t spins = 0;
            bool bad = false;
            unsigned long long w = 0;
            if (has_peer) {
                while (((w = ld_relaxed_sys(&mine->min_next[lane])) >> 32) != epoch) {
                    if ((++spins & 1023u) == 0 && (*(volatile uint32_t *)&st->error || pglobal_ns() - t0 > kPeelWatchdogNs)) { bad = true; break; }
                }
                gmin = (int32_t)((uint32_t)w & 0x7fffffffu);
                any_active = ((uint32_t)w & 0x80000000u) != 0;
            }
            if (__ballot_sync(kFullMask, bad)) { if (lane == 0) atomicCAS(&st->error, 0u, (uint32_t)kErrPeers); failed = true; break; }
            gmin = warp_reduce_min(gmin);
            any_active = __any_sync(kFullMask, any_active);
        }
        if (any_active && lane == 0) {   // the level that just ended peeled something somewhere: it counts
            st->levels += 1;
            st->max_core = prev_k;
        }
        KG_APROF(1);
        if (gmin == INT32_MAX) break;   // nothing alive anywhere
        const int32_t k = gmin;
        // ---- scan: the level's first unitigs into the pool, survivors compacted
        const uint32_t dst = src == 0u ? 1u : 0u;
        if (lane == 0) {
            st->cur_k = k;
            st->n_alive = n_alive;     // the list the scan reads (the survivors of the previous scan) ...
            st->alive_src = src;
            st->alive_cnt[dst] = 0;    // ... and the one it writes
        }
        __syncwarp();
        if (!a_issue_and_wait(R, st, seq, kPhScan, k, phases_run, true)) { failed = true; break; }
        if (lane == 0) n_alive = *(volatile uint32_t *)&st->alive_cnt[dst];
        n_alive = __shfl_sync(kFullMask, n_alive, 0);
        src = dst;
        prev_k = k;
        KG_APROF(2);
        // ---- nobody decrements before every rank's scan is complete
        if (has_peer) st_relaxed_sys(&R.ctl_peer[lane]->scan_seen[R.rank], epoch);
        {
            const unsigned long long t0 = pglobal_ns();
            uint32_t spins = 0;
            bool bad = false;
            if (has_peer) {
                while (ld_relaxed_sys(&mine->scan_seen[lane]) != epoch) {
                    if ((++spins & 1023u) == 0 && (*(volatile uint32_t *)&st->error || pglobal_ns() - t0 > kPeelWatchdogNs)) { bad = true; break; }
                }
            }
            if (__ballot_sync(kFullMask, bad)) { if (lane == 0) atomicCAS(&st->error, 0u, (uint32_t)kErrPeers); failed = true; break; }
        }
        KG_APROF(3);
        a_issue_and_wait(R, st, seq, kPhGo, k, phases_run, false);
        unsigned long long done_before = lane == 0 ? ld_relaxed_sys(&mine->q_done) : 0ull;
        done_before = __shfl_sync(kFullMask, done_before, 0);
        // ---- the end of the level: every rank idle at one instant
        {
            const unsigned long long t0 = pglobal_ns();
            uint32_t spins = 0;
            while (true) {
                unsigned long long d1 = 0, t1 = 0, t2 = 0;
                if (has_peer) {
                    d1 = ld_relaxed_sys(&R.ctl_peer[lane]->q_done);    // done first: done <= tail at any instant
                    t1 = ld_relaxed_sys(&R.ctl_peer[lane]->q_tail);
                }
                if (__all_sync(kFullMask, d1 == t1)) {
                    if (has_peer) t2 = ld_relaxed_sys(&R.ctl_peer[lane]->q_tail);
                    if (__all_sync(kFullMask, t2 == t1)) break;
                }
                if ((++spins & 255u) == 0) {
                    const bool bad = *(volatile uint32_t *)&st->error || pglobal_ns() - t0 > kPeelWatchdogNs;
                    if (__any_sync(kFullMask, bad)) { if (lane == 0) atomicCAS(&st->error, 0u, (uint32_t)kErrPeers); failed = true; break; }
                }
            }
            unsigned long long done_after = lane == 0 ? ld_relaxed_sys(&mine->q_done) : 0ull;
            done_after = __shfl_sync(kFullMask, done_after, 0);
            level_active = done_after != done_before;
            if (lane == 0 && epoch <= (unsigned long long)kALvlProf) {
                st->lvl_ns[epoch - 1] = (uint32_t)(pglobal_ns() - t0);
                st->lvl_k[epoch - 1] = k;
                st->lvl_pushed[epoch - 1] = (uint32_t)(done_after - done_before);
            }
        }
        KG_APROF(4);
    }
#undef KG_APROF
    a_issue_and_wait(R, st, seq, kPhExit, -1, phases_run, false);
}

__global__ void __launch_bounds__(kAThreads, 2) apeel_kernel(const ARank *ranks, uint32_t ctas_per_rank) {
    __shared__ uint32_t s_scan[kAWarps + 1];
    __shared__ uint32_t s_base[2];
    __shared__ unsigned long long s_base64;
    __shared__ ARank s_rank;   // the per-rank pointer tables are indexed by owner: shared memory, not a register copy
    if (threadIdx.x == 0) s_rank = ranks[blockIdx.x / ctas_per_rank];
    __syncthreads();
    const ARank &R = s_rank;
    const uint32_t cta = blockIdx.x % ctas_per_rank;
    if (cta == 0) {
        if (threadIdx.x < 32) a_manager(R);
        return;
    }
    a_worker(R, cta - 1u, R.ctas - 1u, s_scan, s_base, &s_base64);
}

}  // namespace

int dist_peel_async(kombgpu_dist_graph *g, int rc) {
    kombgpu_comm *c = g->comm;
    kombgpu_ctx *ctx = g->ctx;
    const int world = c->world;
    const uint32_t n_local = g->n_local;
    if (!g->row_ptr32) return ctx_fail(ctx, KOMBGPU_ESTATE, "the asynchronous peel needs the rank's rows (built with the async layout)");

    // symmetric: working degrees, pool, control block, map of peeled unitigs (one byte per unitig of the graph on every
    // rank).  The pool holds every local unitig once plus the slices of long rows; all ranks size it alike (the symmetric
    // heap hands out the same sequence of buffers everywhere).
    unsigned long long mine_sz[1] = {(unsigned long long)n_local + g->n_directed / kASlice + 64ull}, all_sz[kMaxRanks];
    KG_TRY(exchange_rc(c, rc, mine_sz, 1, all_sz));
    unsigned long long cap64 = 0;
    for (int q = 0; q < world; ++q) cap64 = all_sz[q] > cap64 ? all_sz[q] : cap64;
    if (cap64 >= 0xffffffffull) return ctx_fail(ctx, KOMBGPU_EINVAL, "partition too large for the peel's pool");   // on every rank
    SymRewind heap{c, sym_mark(c)};
    int32_t *work = nullptr;
    unsigned long long *pool = nullptr;
    ACtl *ctl = nullptr;
    uint8_t *dead = nullptr;
    PeerPtrs<int32_t> work_peers{};
    PeerPtrs<unsigned long long> pool_peers{};
    PeerPtrs<ACtl> ctl_peers{};
    PeerPtrs<uint8_t> dead_peers{};
    rc = first_rc(rc, sym_alloc(c, (size_t)g->step, &work, &work_peers));
    rc = first_rc(rc, sym_alloc(c, (size_t)cap64, &pool, &pool_peers));
    rc = first_rc(rc, sym_alloc(c, 1, &ctl, &ctl_peers));
    rc = first_rc(rc, sym_alloc(c, (size_t)g->n_global, &dead, &dead_peers));

    DevBuf<uint32_t> alive_a, alive_b;
    DevBuf<AState> state;
    DevBuf<ARank> desc;
    uint32_t ctas_per_rank = 0;
    ARank R{};
    if (rc == KOMBGPU_OK) rc = [&]() -> int {
        KG_CUDA(ctx, cudaMemsetAsync(g->core, 0, (size_t)(n_local ? n_local : 1) * sizeof(int32_t), ctx->stream));
        KG_CUDA(ctx, cudaMemsetAsync(dead, 0, (size_t)(g->n_global ? g->n_global : 1), ctx->stream));
        KG_CUDA(ctx, cudaMemsetAsync(ctl, 0, sizeof(ACtl), ctx->stream));
        KG_CUDA(ctx, cudaMemsetAsync(pool, 0xff, (size_t)cap64 * sizeof(unsigned long long), ctx->stream));
        if (n_local) KG_CUDA(ctx, cudaMemcpyAsync(work, g->deg, (size_t)n_local * sizeof(int32_t), cudaMemcpyDeviceToDevice, ctx->stream));
        KG_ALLOC(ctx, alive_a, n_local);
        KG_ALLOC(ctx, alive_b, n_local);
        KG_ALLOC(ctx, state, 1);
        KG_ALLOC(ctx, desc, kMaxRanks);
        KG_CUDA(ctx, cudaMemsetAsync(state.p, 0, sizeof(AState), ctx->stream));
        KG_TRY(rank_ctas(ctx, c, apeel_kernel, kAThreads, 2, &ctas_per_rank));   // CTA 0 manages, the others work
        R.n_local = n_local; R.v_lo = g->v_lo; R.n_global = g->n_global; R.step = g->step; R.world = world; R.rank = c->rank;
        R.ctas = ctas_per_rank;
        R.row_ptr = g->row_ptr32; R.col = g->col; R.core = g->core;
        R.alive[0] = alive_a.p; R.alive[1] = alive_b.p;
        R.pool_cap = (uint32_t)cap64;
        for (int q = 0; q < world; ++q) {
            R.deg_peer[q] = work_peers.p[q];
            R.pool_peer[q] = pool_peers.p[q];
            R.ctl_peer[q] = ctl_peers.p[q];
            R.dead_peer[q] = dead_peers.p[q];
        }
        R.st = state.p;
        return KOMBGPU_OK;
    }();
    // every rank's degrees, pool and control words are initialised before anyone reaches into them
    KG_TRY(barrier_rc(c, rc));

    const cudaError_t le = launch_ranks(c, apeel_kernel, kAThreads, ctas_per_rank, R, desc.p, nullptr);
    if (le != cudaSuccess) rc = ctx_fail(ctx, KOMBGPU_ECUDA, "asynchronous peel kernel: %s", cudaGetErrorString(le));
    AState fin{};
    ACtl fin_ctl{};
    if (rc == KOMBGPU_OK) rc = read_back(ctx, state.p, &fin, 1);
    if (rc == KOMBGPU_OK) rc = read_back(ctx, ctl, &fin_ctl, 1);
    // global figures; also: nobody gives back its pool (at return) while a peer may still be writing
    const unsigned long long peeled_here = fin_ctl.q_done - fin.n_slices;
    unsigned long long mine[3] = {fin.error, peeled_here, (unsigned long long)(uint32_t)fin.max_core}, all[kMaxRanks * 3];
    KG_TRY(exchange_rc(c, rc, mine, 3, all));
    uint64_t peeled = 0;
    for (int q = 0; q < world; ++q) {
        if (all[q * 3]) return ctx_fail(ctx, KOMBGPU_EINTERNAL, "asynchronous peel: rank %d reports error %llu (%s)", q, all[q * 3], rank_error_text(all[q * 3]));
        peeled += all[q * 3 + 1];
    }
    if (peeled != g->n_global) return ctx_fail(ctx, KOMBGPU_EINTERNAL, "asynchronous peel ended with %llu of %u unitigs peeled", (unsigned long long)peeled, g->n_global);
    g->st.max_coreness = fin.max_core;
    g->st.peel_levels = fin.levels;
    g->st.peel_subrounds = fin.levels;          // the ranks meet once per level here, not once per cascade generation
    g->st.peel_solo_subrounds = 0;
    g->st.peel_async = 1;
    g->st.n_messages_sent = fin.n_remote_push;               // unitigs this rank discovered for other ranks (pushed into their pools)
    g->st.n_messages_recv = fin_ctl.q_tail - fin.n_own_push;   // unitigs other ranks pushed into this rank's pool
    if (getenv("KOMBGPU_DEBUG"))
        fprintf(stderr, "[kombgpu] rank %d apeel: levels %u ctas %u | manager ms: min pass %.3f min exchange %.3f scan pass %.3f scan exchange %.3f "
                "levels (go -> over) %.3f | peeled here %llu, slices %llu, entries visited %llu, remote decrements %llu, remote pushes %llu\n",
                c->rank, fin.levels, ctas_per_rank, fin.prof_ns[0] * 1e-6, fin.prof_ns[1] * 1e-6, fin.prof_ns[2] * 1e-6, fin.prof_ns[3] * 1e-6,
                fin.prof_ns[4] * 1e-6, peeled_here, fin.n_slices, fin.n_visited, fin.n_remote_dec, fin.n_remote_push);
    if (getenv("KOMBGPU_DEBUG") && c->rank == 0) {
        fprintf(stderr, "[kombgpu] apeel levels (k: us from go to over / entries processed on rank 0):");
        for (uint32_t i = 0; i < fin.levels && i < (uint32_t)kALvlProf; ++i) fprintf(stderr, " %d:%.0f/%u", fin.lvl_k[i], fin.lvl_ns[i] * 1e-3, fin.lvl_pushed[i]);
        fprintf(stderr, "\n");
    }
    return KOMBGPU_OK;
}

}  // namespace kg
