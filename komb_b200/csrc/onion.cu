// onion.cu — the onion decomposition (Hébert-Dufresne, Grochow & Allard, Sci. Rep. 6:31708, 2016): every k-shell
// split into the layers of a synchronous peel, as networkx.onion_layers defines them.
//
// Degree-0 vertices form layer 1 when there are any.  Then, with k = max(k, smallest remaining degree), the next layer
// is every remaining vertex whose remaining degree is <= k, and the whole layer is removed at once.  Layer l + 1 may
// only be formed once every decrement caused by layer l has landed, so this is a peel whose generations are exact;
// the k-core peel (peel.cu) lets cascade generations mix on purpose and cannot give this order.
//
// One persistent cooperative kernel runs the whole decomposition, with no host round trip per layer:
//   level k:  SCAN   one pass over the compacted alive list: vertices with deg == k are the level's first layer,
//                    vertices above k are compacted, the rest (removed earlier) are dropped; the survivors' minimum
//                    degree is the next level when this one turns out empty
//             LAYERS the layer [lb, le) of order[] walks its rows and decrements every neighbour; the thread whose
//                    decrement takes a degree from k + 1 to k owns that vertex and appends it to order[] as the next
//                    layer.  Degrees are never clamped: a vertex already at or below k (in this layer or removed
//                    earlier) can never make that step again, so each vertex enters order[] exactly once.
// A layer of at most kThinV vertices and kThinEdges edges is run by CTA 0 alone, with block barriers, for as many
// consecutive layers as stay thin, while the other CTAs wait at the next grid barrier: a chain of thin layers costs
// no grid barrier per layer.  Wider layers go to the whole grid: vertices in tiles spread over every CTA, rows longer than kSplit as slices
// of kSliceLen edges, which every CTA takes after one more grid barrier -- so a hub's decrements also land inside
// its layer.  The kernel has no spin of its own: its only waits are grid barriers.
#include <cooperative_groups.h>

#include "graph.cuh"
#include "kombgpu_debug.h"

namespace cg = cooperative_groups;

namespace kg {
namespace {

constexpr int kOnionThreads = 512;
constexpr int kOnionWarps = kOnionThreads / 32;
constexpr uint32_t kThinV = kOnionThreads;   // a thin layer: one vertex per thread of CTA 0 ...
constexpr uint32_t kThinEdges = 16384;       // ... and at most this many edges
constexpr uint32_t kSplit = 2048;            // rows longer than this are cut into slices shared by all CTAs
constexpr uint32_t kSliceLen = 2048;
constexpr int kUnroll = 4;                   // independent col -> atomic chains per thread
constexpr int kScanItems = 8;                // alive-list entries per thread per scan tile

enum : uint32_t { kErrOrderFull = 1, kErrSliceFull = 2 };

// Counters of one step (a scan, a thin run or a wide layer), in three rotating slots: step s uses slot s % 3 and CTA 0
// re-arms slot (s + 1) % 3 when step s starts.  Every step ends at a grid barrier and its slot is read between that
// barrier and the next one, so slot (s + 1) % 3, last read in step s - 2, is free, and nobody writes it before the
// barrier that ends step s.  Every decision that leads to a grid barrier is taken from a slot or from values that are
// only written a barrier or more away, so all CTAs take the same path to the same barriers.
struct StepSlot {
    uint32_t found;       // vertices appended as the next layer (the scan: the level's first layer)
    uint32_t slices;      // slices published (wide layers)
    uint32_t alive_out;   // survivors the scan compacted
    int32_t next_min;     // their smallest degree
};
struct OnionState {
    StepSlot slot[3];
    uint32_t lb, le, layer; // the thin run's hand-back: the pending layer [lb, le) and its number (the last non-empty
    uint32_t wide;          // layer's when the range is empty); wide = 1: the pending layer goes to the whole grid
    uint32_t error;         // reported to the host; never steers the kernel, which always runs to its end
    uint32_t placed, n_layers, levels, steps, thin_layers;
};

struct OnionShared {
    uint32_t list[2][kThinV];   // the thin run's current / next layer
    uint64_t row[kOnionThreads];
    uint32_t off[kOnionThreads + 1];
    uint32_t scan[kOnionWarps + 1];
    uint32_t tile_base[2];
    uint32_t cnt;               // the thin run's discoveries in the current layer
    uint32_t ctl;
};

// The thread whose decrement took deg[u] from k + 1 to k appends u: warp-aggregated position from *ctr, entry at
// order[base + pos] with its layer number and coreness k.  thin_next (CTA 0's run): the first kThinV positions also go to shared memory.
// Called by whole warps.
__device__ __forceinline__ void push_found(bool p, uint32_t u, uint32_t *ctr, uint32_t base, uint32_t n, uint32_t *order,
                                           uint32_t *layer, int32_t *core, int32_t k, uint32_t lnext, uint32_t *thin_next, uint32_t *err) {
    const uint32_t m = __ballot_sync(kFullMask, p);
    if (m == 0) return;
    uint32_t pos = 0;
    if (lane_id() == 0) pos = atomicAdd(ctr, (uint32_t)__popc(m));
    pos = __shfl_sync(kFullMask, pos, 0) + __popc(m & lanemask_lt());
    if (!p) return;
    const uint32_t at = base + pos;
    if (at < n) {
        order[at] = u;
        layer[u] = lnext;
        core[u] = k;
    } else {
        atomicExch(err, kErrOrderFull);
    }
    if (thin_next && pos < kThinV) thin_next[pos] = u;
}

// Decrement the far end of every edge of the batch in sh.row / sh.off (up to kOnionThreads ranges, `total` edges) and
// append the vertices that reach k.  Every thread keeps kUnroll independent chains in flight.
__device__ __forceinline__ void relax_batch(uint32_t total, int32_t k, const uint32_t *__restrict__ col, int32_t *deg,
                                            uint32_t *ctr, uint32_t base, uint32_t n, uint32_t *order, uint32_t *layer, int32_t *core,
                                            uint32_t lnext, uint32_t *thin_next, uint32_t *err, const OnionShared &sh) {
    const uint32_t tid = threadIdx.x;
    for (uint32_t b = 0; b < total; b += kOnionThreads * kUnroll) {
        uint32_t u[kUnroll];
        int32_t d[kUnroll];
#pragma unroll
        for (int t = 0; t < kUnroll; ++t) {
            const uint32_t e = b + t * kOnionThreads + tid;
            u[t] = kFullMask;
            if (e < total) {
                uint32_t lo = 0, hi = kOnionThreads;   // off[lo] <= e < off[hi]: the last range that starts at or before e
#pragma unroll
                for (int s = 0; s < 9; ++s) {
                    const uint32_t mid = (lo + hi) >> 1;
                    if (sh.off[mid] <= e) lo = mid; else hi = mid;
                }
                u[t] = col[sh.row[lo] + (e - sh.off[lo])];
            }
        }
#pragma unroll
        for (int t = 0; t < kUnroll; ++t) d[t] = u[t] != kFullMask ? atomicSub(&deg[u[t]], 1) : INT32_MIN;
#pragma unroll
        for (int t = 0; t < kUnroll; ++t) push_found(d[t] == k + 1, u[t], ctr, base, n, order, layer, core, k, lnext, thin_next, err);
    }
}

// one slice of a long row, by the whole CTA
__device__ __forceinline__ void relax_slice(uint64_t first, uint32_t len, int32_t k, const uint32_t *__restrict__ col, int32_t *deg,
                                            uint32_t *ctr, uint32_t base, uint32_t n, uint32_t *order, uint32_t *layer, int32_t *core,
                                            uint32_t lnext, uint32_t *err) {
    for (uint32_t b = 0; b < len; b += kOnionThreads * kUnroll) {
        uint32_t u[kUnroll];
        int32_t d[kUnroll];
#pragma unroll
        for (int t = 0; t < kUnroll; ++t) {
            const uint32_t e = b + t * kOnionThreads + threadIdx.x;
            u[t] = e < len ? col[first + e] : kFullMask;
        }
#pragma unroll
        for (int t = 0; t < kUnroll; ++t) d[t] = u[t] != kFullMask ? atomicSub(&deg[u[t]], 1) : INT32_MIN;
#pragma unroll
        for (int t = 0; t < kUnroll; ++t) push_found(d[t] == k + 1, u[t], ctr, base, n, order, layer, core, k, lnext, nullptr, err);
    }
}

// SCAN of level k for one CTA: deg == k -> order[base + ...] (layer lnum), deg > k -> alive_dst, the rest dropped.
// Positions come from a CTA-wide scan: two global atomics per tile.  Returns the thread's minimum survivor degree.
__device__ __forceinline__ int32_t onion_scan(int32_t k, uint32_t lnum, const uint32_t *alive_src, uint32_t n_alive, uint32_t *alive_dst,
                                              const int32_t *deg, uint32_t base, uint32_t n, uint32_t *order, uint32_t *layer,
                                              int32_t *core, StepSlot *slot, uint32_t *err, OnionShared &sh) {
    const uint32_t tid = threadIdx.x;
    int32_t local_min = INT32_MAX;
    // short lists are spread over all CTAs (see peel_device.cuh scan_alive)
    const uint32_t per_cta = (uint32_t)(((uint64_t)n_alive + gridDim.x - 1) / gridDim.x);
    const int items = (int)min(max((per_cta + kOnionThreads - 1) / kOnionThreads, 1u), (uint32_t)kScanItems);
    const uint64_t tile_v = (uint64_t)items * kOnionThreads;
    for (uint64_t tile = (uint64_t)blockIdx.x * tile_v; tile < n_alive; tile += (uint64_t)gridDim.x * tile_v) {
        uint32_t v[kScanItems], flag[kScanItems];   // 1 = this level's first layer, 0x10000 = survivor
        uint32_t mine = 0;
#pragma unroll
        for (int j = 0; j < kScanItems; ++j) {
            const uint64_t i = (j < items) ? tile + (uint64_t)j * kOnionThreads + tid : ~0ull;
            flag[j] = 0;
            v[j] = 0;
            if (i < n_alive) v[j] = alive_src ? __ldcg(&alive_src[i]) : (uint32_t)i;
        }
#pragma unroll
        for (int j = 0; j < kScanItems; ++j) {
            const uint64_t i = (j < items) ? tile + (uint64_t)j * kOnionThreads + tid : ~0ull;
            if (i < n_alive) {
                const int32_t d = __ldcg(&deg[v[j]]);
                if (d == k) flag[j] = 1u;
                else if (d > k) { flag[j] = 0x10000u; local_min = min(local_min, d); }
            }
            mine += flag[j];
        }
        uint32_t total = 0;
        const uint32_t ex = block_excl_scan_add<uint32_t, kOnionThreads>(mine, sh.scan, &total);   // both counts, 16 bits each
        if (tid == 0) {
            const uint32_t nf = total & 0xffffu, ns = total >> 16;
            sh.tile_base[0] = nf ? atomicAdd(&slot->found, nf) : 0;
            sh.tile_base[1] = ns ? atomicAdd(&slot->alive_out, ns) : 0;
        }
        __syncthreads();
        uint32_t fpos = base + sh.tile_base[0] + (ex & 0xffffu), spos = sh.tile_base[1] + (ex >> 16);
#pragma unroll
        for (int j = 0; j < kScanItems; ++j) {
            if (flag[j] == 1u) {
                if (fpos < n) { order[fpos] = v[j]; layer[v[j]] = lnum; core[v[j]] = k; }
                else atomicExch(err, kErrOrderFull);
                ++fpos;
            } else if (flag[j]) {
                alive_dst[spos++] = v[j];
            }
        }
        __syncthreads();   // tile_base is reused by the next tile
    }
    return local_min;
}

// CTA 0 alone: layer [lb, le) (number lnum, le - lb <= kThinV) and the layers after it while they stay thin.  Hands the
// first layer it does not run back through st: its range and number with wide = 1, or an empty range and the number of
// the last layer it ran when the level is over.
__device__ __forceinline__ void thin_run(int32_t k, uint32_t lb, uint32_t le, uint32_t lnum, uint32_t n, const uint64_t *__restrict__ row_ptr,
                         const uint32_t *__restrict__ col, int32_t *deg, uint32_t *order, uint32_t *layer, int32_t *core, OnionState *st,
                         OnionShared &sh) {
    const uint32_t tid = threadIdx.x;
    uint32_t cur = 0, ran = 0, wide = 0;
    bool from_order = true;    // the first layer is read from order[], the next ones from shared memory
    while (true) {
        const uint32_t size = le - lb;
        uint64_t row = 0;
        uint32_t len = 0;
        if (size <= kThinV && tid < size) {
            const uint32_t v = from_order ? __ldcg(&order[lb + tid]) : sh.list[cur][tid];
            // a row longer than kThinEdges sends the layer to the grid on its own; clamped, the sum cannot wrap
            row = row_ptr[v];
            len = (uint32_t)min(row_ptr[v + 1] - row, (uint64_t)kThinEdges + 1);
        }
        uint32_t total = 0;
        const uint32_t ex = block_excl_scan_add<uint32_t, kOnionThreads>(len, sh.scan, &total);
        if (size > kThinV || total > kThinEdges) { wide = 1; break; }
        sh.off[tid] = ex;
        sh.row[tid] = row;
        if (tid == 0) { sh.off[kOnionThreads] = total; sh.cnt = 0; }
        __syncthreads();
        relax_batch(total, k, col, deg, &sh.cnt, le, n, order, layer, core, lnum + 1, sh.list[cur ^ 1], &st->error, sh);
        __syncthreads();
        const uint32_t found = min(sh.cnt, n - le);   // more would be a broken invariant, flagged by push_found
        __syncthreads();   // everyone has read cnt before the next layer resets it
        ++ran;
        from_order = false;
        cur ^= 1;
        lb = le;
        le += found;
        if (found == 0) break;   // the level is over
        ++lnum;
    }
    if (tid == 0) {
        st->lb = lb; st->le = le; st->layer = lnum; st->wide = wide;
        st->thin_layers += ran;
    }
}

__global__ void __launch_bounds__(kOnionThreads, 1) onion_kernel(uint32_t n, const uint64_t *__restrict__ row_ptr, const uint32_t *__restrict__ col,
                                                              int32_t *deg, uint32_t *layer, int32_t *core, uint32_t *order, uint32_t *alive_a, uint32_t *alive_b,
                                                              uint64_t *sl_first, uint32_t *sl_len, uint32_t sl_cap, OnionState *st) {
    cg::grid_group grid = cg::this_grid();
    __shared__ OnionShared sh;
    const uint32_t tid = threadIdx.x;
    const bool boss = blockIdx.x == 0 && tid == 0;

    int32_t k = 0;
    uint32_t n_alive = n, lnum = 0;           // lnum: the number of the last non-empty layer
    uint32_t placed = 0;                      // vertices in order[]
    const uint32_t *alive_src = nullptr;      // nullptr = identity (every vertex)
    uint32_t *alive_dst = alive_a;
    uint32_t step = 0, slices_done = 0;
    auto begin_step = [&]() -> StepSlot * {
        if (boss) {
            StepSlot &x = st->slot[(step + 1) % 3];
            x.found = 0; x.slices = 0; x.alive_out = 0; x.next_min = INT32_MAX;
            st->steps = step + 1;
        }
        return &st->slot[step % 3];
    };

    while (true) {
        StepSlot *slot = begin_step();
        int32_t mn = onion_scan(k, lnum + 1, alive_src, n_alive, alive_dst, deg, placed, n, order, layer, core, slot, &st->error, sh);
        mn = warp_reduce_min(mn);
        if (lane_id() == 0 && mn != INT32_MAX) atomicMin(&slot->next_min, mn);
        grid.sync();
        ++step;
        const uint32_t front = min(__ldcg(&slot->found), n - placed), survivors = __ldcg(&slot->alive_out);
        const int32_t min_next = __ldcg(&slot->next_min);
        alive_src = alive_dst;
        alive_dst = alive_dst == alive_a ? alive_b : alive_a;
        n_alive = survivors;
        if (front == 0) {
            if (survivors == 0 || min_next == INT32_MAX) break;
            k = min_next;   // no vertex at k: the next level is the smallest remaining degree
            continue;
        }
        uint32_t lb = placed, le = placed + front;
        ++lnum;
        if (boss) st->levels += 1;
        bool wide = front > kThinV;
        while (true) {
            slot = begin_step();
            if (!wide) {
                if (blockIdx.x == 0) thin_run(k, lb, le, lnum, n, row_ptr, col, deg, order, layer, core, st, sh);
                grid.sync();
                ++step;
                lb = __ldcg(&st->lb); le = __ldcg(&st->le); lnum = __ldcg(&st->layer); wide = __ldcg(&st->wide) != 0;
                if (lb == le) break;   // the level is over
                continue;
            }
            // the whole grid: the layer dealt out in tiles of up to kOnionThreads vertices, small enough that every
            // CTA gets one when the layer allows it; long rows become slices
            const uint32_t tile = min((uint32_t)kOnionThreads, max(1u, (le - lb + gridDim.x - 1) / gridDim.x));
            for (uint64_t t0 = lb + (uint64_t)blockIdx.x * tile; t0 < le; t0 += (uint64_t)gridDim.x * tile) {
                const uint64_t i = t0 + tid;
                uint64_t row = 0;
                uint32_t len = 0;
                if (tid < tile && i < le) {
                    const uint32_t v = __ldcg(&order[i]);
                    row = row_ptr[v];
                    len = (uint32_t)(row_ptr[v + 1] - row);
                    if (len > kSplit) {
                        const uint32_t ns = (len + kSliceLen - 1) / kSliceLen;
                        const uint32_t s0 = slices_done + atomicAdd(&slot->slices, ns);
                        if (s0 + ns <= sl_cap) {
                            for (uint32_t s = 0; s < ns; ++s) {
                                sl_first[s0 + s] = row + (uint64_t)s * kSliceLen;
                                sl_len[s0 + s] = min(kSliceLen, len - s * kSliceLen);
                            }
                        } else {
                            atomicExch(&st->error, kErrSliceFull);
                        }
                        len = 0;
                    }
                }
                uint32_t total = 0;
                const uint32_t ex = block_excl_scan_add<uint32_t, kOnionThreads>(len, sh.scan, &total);
                sh.off[tid] = ex;
                sh.row[tid] = row;
                if (tid == 0) sh.off[kOnionThreads] = total;
                __syncthreads();
                relax_batch(total, k, col, deg, &slot->found, le, n, order, layer, core, lnum + 1, nullptr, &st->error, sh);
                __syncthreads();   // off / row are reused by the next tile
            }
            grid.sync();
            const uint32_t slices = min(__ldcg(&slot->slices), sl_cap - slices_done);
            if (slices) {
                // the slices of this layer's long rows: their decrements also land before the next layer is read
                for (uint32_t s = slices_done + blockIdx.x; s < slices_done + slices; s += gridDim.x)
                    relax_slice(__ldcg(&sl_first[s]), __ldcg(&sl_len[s]), k, col, deg, &slot->found, le, n, order, layer, core, lnum + 1, &st->error);
                slices_done += slices;
                grid.sync();
            }
            ++step;
            const uint32_t found = min(__ldcg(&slot->found), n - le);
            lb = le;
            le += found;
            if (found == 0) break;   // the level is over
            ++lnum;
            wide = found > kThinV;
        }
        placed = le;
        k += 1;
    }
    if (boss) { st->placed = placed; st->n_layers = lnum; }
}

}  // namespace

int onion_layers(kombgpu_graph *g) {
    kombgpu_ctx *ctx = g->ctx;
    const uint32_t n = g->n;
    onion_release(g);
    DevBuf<uint32_t> layer;
    DevBuf<int32_t> core;
    KG_ALLOC(ctx, layer, n);
    KG_ALLOC(ctx, core, n);
    if (n == 0) {
        g->onion_layer = layer.take();
        g->onion_core = core.take();
        g->onion_n_layers = 0;
        g->has_onion = true;
        return KOMBGPU_OK;
    }
    int per_sm = 0;
    KG_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, onion_kernel, kOnionThreads, 0));
    if (per_sm < 1) return ctx_fail(ctx, KOMBGPU_ECUDA, "onion kernel does not fit on an SM");
    const int grid = per_sm * ctx->sm_count;   // persistent: every CTA resident (cooperative launch)

    // each vertex is removed once, so each long row is sliced once: <= 2E / kSplit rows, len / kSliceLen + 1 slices each
    const uint64_t cap64 = 2 * g->n_edges / kSliceLen + 2 * g->n_edges / kSplit + 1;
    if (cap64 >= 0xffffffffull) return ctx_fail(ctx, KOMBGPU_EINVAL, "graph too large for the onion's slice list");
    DevBuf<int32_t> deg;
    DevBuf<uint32_t> order, alive_a, alive_b, sl_len;
    DevBuf<uint64_t> sl_first;
    DevBuf<OnionState> state;
    KG_ALLOC(ctx, deg, n);
    KG_ALLOC(ctx, order, n);
    KG_ALLOC(ctx, alive_a, n);
    KG_ALLOC(ctx, alive_b, n);
    KG_ALLOC(ctx, sl_first, cap64);
    KG_ALLOC(ctx, sl_len, cap64);
    KG_ALLOC(ctx, state, 1);
    KG_CUDA(ctx, cudaMemsetAsync(sl_len.p, 0, cap64 * sizeof(uint32_t), ctx->stream));   // a slice never written is empty
    KG_CUDA(ctx, cudaMemcpyAsync(deg.p, g->deg, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToDevice, ctx->stream));
    OnionState init{};
    for (int i = 0; i < 3; ++i) init.slot[i].next_min = INT32_MAX;
    KG_CUDA(ctx, cudaMemcpyAsync(state.p, &init, sizeof(init), cudaMemcpyHostToDevice, ctx->stream));

    uint32_t n_arg = n, cap_arg = (uint32_t)cap64;
    const uint64_t *row_ptr = g->row_ptr;
    const uint32_t *col = g->col;
    int32_t *dp = deg.p, *cp = core.p;
    uint32_t *lp = layer.p, *op = order.p, *aa = alive_a.p, *ab = alive_b.p, *slp = sl_len.p;
    uint64_t *sfp = sl_first.p;
    OnionState *sp = state.p;
    void *args[] = {&n_arg, &row_ptr, &col, &dp, &lp, &cp, &op, &aa, &ab, &sfp, &slp, &cap_arg, &sp};
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    KG_CUDA(ctx, cudaEventCreate(&ev0));
    KG_CUDA(ctx, cudaEventCreate(&ev1));
    cudaEventRecord(ev0, ctx->stream);
    cudaError_t le = cudaLaunchCooperativeKernel((void *)onion_kernel, dim3(grid), dim3(kOnionThreads), args, 0, ctx->stream);
    cudaEventRecord(ev1, ctx->stream);
    ctx->launches++;
    if (le == cudaSuccess) le = cudaEventSynchronize(ev1);
    float ms = 0.f;
    if (le == cudaSuccess) cudaEventElapsedTime(&ms, ev0, ev1);
    cudaEventDestroy(ev0);
    cudaEventDestroy(ev1);
    if (le != cudaSuccess) return ctx_fail(ctx, KOMBGPU_ECUDA, "onion kernel: %s", cudaGetErrorString(le));

    OnionState fin{};
    KG_TRY(read_back(ctx, state.p, &fin, 1));
    if (fin.error) return ctx_fail(ctx, KOMBGPU_EINTERNAL, "onion invariant broken (code %u, %u of %u vertices placed)", fin.error, fin.placed, n);
    if (fin.placed != n) return ctx_fail(ctx, KOMBGPU_EINTERNAL, "onion ended with %u of %u vertices placed", fin.placed, n);
    g->onion_layer = layer.take();
    g->onion_core = core.take();
    g->onion_n_layers = fin.n_layers;
    g->onion_info = OnionInfo{ms, fin.levels, fin.steps, fin.thin_layers};
    g->has_onion = true;
    return KOMBGPU_OK;
}

void onion_release(kombgpu_graph *g) {
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

int kombgpu_graph_onion(kombgpu_graph *g, uint32_t *layer, uint32_t *n_layers) {
    if (!g) return KOMBGPU_EINVAL;
    kombgpu_ctx *ctx = g->ctx;
    KG_CUDA(ctx, cudaSetDevice(ctx->device));
    if (!g->has_onion) {
        const uint64_t launches0 = ctx->launches;
        const int rc = onion_layers(g);
        g->st.kernel_launches += ctx->launches - launches0;
        if (rc != KOMBGPU_OK) return rc;
    }
    if (n_layers) *n_layers = g->onion_n_layers;
    if (layer && g->n) {
        KG_CUDA(ctx, cudaMemcpyAsync(layer, g->onion_layer, (size_t)g->n * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
        KG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return KOMBGPU_OK;
}

// measurement aids (include/kombgpu_debug.h)
int kombgpu_debug_onion_again(kombgpu_graph *g) {
    if (!g) return KOMBGPU_EINVAL;
    g->has_onion = false;
    return kombgpu_graph_onion(g, nullptr, nullptr);
}

int kombgpu_debug_onion_timing(const kombgpu_graph *g, float *ms_kernel, uint32_t *levels, uint32_t *steps, uint32_t *thin_layers) {
    if (!g) return KOMBGPU_EINVAL;
    if (!g->has_onion) return ctx_fail(g->ctx, KOMBGPU_ESTATE, "kombgpu_graph_onion has not run");
    if (ms_kernel) *ms_kernel = g->onion_info.ms_kernel;
    if (levels) *levels = g->onion_info.levels;
    if (steps) *steps = g->onion_info.steps;
    if (thin_layers) *thin_layers = g->onion_info.thin_layers;
    return KOMBGPU_OK;
}

}  // extern "C"
