// trrt_edit.cuh -- map edits on the device, and the re-check of planned trees, routes and mission paths against the map
// as it is now.
//
//   grid_edit_kernel       rectangles of pixels set free or blocked in the packed rows (in-place imarray[y0:y1, x0:x1] = v)
//   tile_patch_kernel      the strip entries (trrt_los.cuh) that hold a pixel of an edited rectangle, rebuilt from the rows
//   validate_edges_kernel  each stored RRT edge tested again with the test that admitted it (rrt.py:173-174)
//   validate_chain_kernel  per node, the AND of the edge verdicts along its cameFrom walk, by pointer doubling
//   validate_path_kernel   Theta* routes (search.lineofsight per step) and mission path rows (the edge test per row)
//
// None of them changes what the planning kernels compute: the pixel tests are the device functions the fused RRT
// kernel and theta_kernel call (los_group, arc_blocked), and the strip entries come from the one strip_entry.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "trrt_bike.cuh"
#include "trrt_device.cuh"
#include "trrt_los.cuh"

namespace trrt {

// ---------------------------------------------------------------------------
// Map edits
// ---------------------------------------------------------------------------
struct EditRect {
    int x0, y0, x1, y1, map;
};
// rectangle r ([n][5] = x0, y0, x1, y1, map) clipped to the image; false when it is empty or its map id is outside
// [0, n_maps) (such a rectangle does nothing)
__device__ __forceinline__ bool edit_rect(const int32_t *__restrict__ rects, int64_t r, int n_maps, int side, EditRect &o) {
    const int32_t *v = rects + 5 * r;
    o.x0 = max(v[0], 0); o.y0 = max(v[1], 0); o.x1 = min(v[2], side); o.y1 = min(v[3], side); o.map = v[4];
    return o.x0 < o.x1 && o.y0 < o.y1 && o.map >= 0 && o.map < n_maps;
}

// One phase of an edit: blocked_phase 0 ORs the masks of the free rectangles into the rows, 1 clears the masks of the
// blocked ones.  The launcher runs phase 0 then phase 1 on one stream, so a pixel that a free and a blocked rectangle
// of one call both cover ends blocked, whatever their order and the atomics' order.  A CTA per rectangle, a thread per
// (row, word) of it; masks stop at the clipped x1 <= W, so the padding bits of a row stay 0.
__global__ void grid_edit_kernel(uint32_t *__restrict__ bits, int n_maps, int side, int wpr, const int32_t *__restrict__ rects,
                                 const uint8_t *__restrict__ free_, int64_t n, int blocked_phase) {
    for (int64_t r = blockIdx.x; r < n; r += gridDim.x) {
        EditRect R;
        if ((free_[r] == 0) != (blocked_phase != 0) || !edit_rect(rects, r, n_maps, side, R)) continue;
        const int w0 = R.x0 >> 5, nw = ((R.x1 - 1) >> 5) - w0 + 1, items = (R.y1 - R.y0) * nw; // <= 2^15 * 2^10
        for (int t = threadIdx.x; t < items; t += blockDim.x) {
            const int y = R.y0 + t / nw, w = w0 + t % nw;
            const int lo = max(R.x0 - 32 * w, 0), hi = min(R.x1 - 32 * w, 32); // bits [lo, hi) of word w
            const uint32_t mask = (hi == 32 ? 0xffffffffu : ((1u << hi) - 1u)) & ~((1u << lo) - 1u);
            const size_t idx = ((size_t)R.map * side + y) * wpr + w;
            TRRT_CHECK(w >= 0 && w < wpr && y >= 0 && y < side && idx < (size_t)n_maps * side * wpr);
            if (blocked_phase) atomicAnd(bits + idx, ~mask);
            else atomicOr(bits + idx, mask);
        }
    }
}

// After both phases: every strip entry that holds a pixel of an edited rectangle, rebuilt from the edited rows.  In
// orientation 0 entry (K, c) holds x in [8c, 8c+8) and y in [8K-8, 8K+8), so the rectangle touches c in
// [x0/8, (x1-1)/8] and K in [y0/8, (y1-1)/8 + 1]; orientation 1 is the same with x and y swapped.  An entry that two
// rectangles touch is written twice with the same value.
__global__ void tile_patch_kernel(const uint32_t *__restrict__ bits, int n_maps, int side, int wpr, int tp, const int32_t *__restrict__ rects,
                                  int64_t n, uint4 *__restrict__ tiles) {
    const size_t epo = (size_t)(tp + 1) * tp;
    for (int64_t r = blockIdx.x; r < n; r += gridDim.x) {
        EditRect R;
        if (!edit_rect(rects, r, n_maps, side, R)) continue;
        const int cx0 = R.x0 >> 3, ncx = ((R.x1 - 1) >> 3) - cx0 + 1, cy0 = R.y0 >> 3, ncy = ((R.y1 - 1) >> 3) - cy0 + 1;
        const int n0 = (ncy + 1) * ncx, n1 = (ncx + 1) * ncy; // entries of orientation 0 and 1
        const uint32_t *src = bits + (size_t)R.map * side * wpr;
        for (int t = threadIdx.x; t < n0 + n1; t += blockDim.x) {
            const int orient = t >= n0, tt = orient ? t - n0 : t, nc = orient ? ncy : ncx;
            const int K = (orient ? cx0 : cy0) + tt / nc, c = (orient ? cy0 : cx0) + tt % nc;
            TRRT_CHECK(K >= 0 && K <= tp && c >= 0 && c < tp);
            tiles[(size_t)R.map * 2 * epo + (orient ? epo : 0) + (size_t)K * tp + c] = strip_entry(src, side, wpr, tp, orient, K, c);
        }
    }
}

// ---------------------------------------------------------------------------
// Validation
// ---------------------------------------------------------------------------
// The edge test of rrt.py:173-174 for the edge (bx, by) -> (lx, ly) with u = (steer, iccx, iccy, rad) as cameFrom stores
// it: search.getArc's pixels on the curve, or the Bresenham line between the int-truncated endpoints for a straight u
// (NaN icc / rad).  Exactly the calls of arc_batch_kernel and of the fused kernel's expansion.  Group-uniform.
template <int G>
__device__ __forceinline__ bool edge_free(const Group<G> &g, const Grid &m, double bx, double by, double lx, double ly, double usteer,
                                          double iccx, double iccy, double rad) {
    if (isnan(iccx) || isnan(rad)) return los_group<G>(g, m, trunc_ll(bx), trunc_ll(by), trunc_ll(lx), trunc_ll(ly));
    return !arc_blocked<G>(g, m, bx, by, lx, ly, usteer, iccx, iccy, rad, nullptr, nullptr);
}

// grid of map `map` (false when the id is outside [0, n_maps): nothing on it is valid)
__device__ __forceinline__ bool map_grid(const uint32_t *bits, int n_maps, int side, int wpr, int map, Grid &m) {
    m.W = side; m.H = side; m.wpr = wpr;
    m.bits = bits + (size_t)(map >= 0 && map < n_maps ? map : 0) * side * wpr;
    return map >= 0 && map < n_maps;
}

struct TreeDev {
    const uint32_t *bits;
    int n_maps, side, wpr, K;
    const int32_t *map_id;
    int64_t nq;
    const double *nx, *ny, *u;
    const int32_t *parent, *n_nodes, *sol;
    uint8_t *edge_ok, *node_ok;
    int8_t *sol_ok;
    int32_t *work; // [nq][3][K]: two (jump, AND) tables and the walk position
};

// edge_ok for every (q, i) of the batch, G lanes per edge, grid-stride so that long and short trees share the SMs.
// Node i's edge is the one from parent[i] with u[i]; 1 for a node without a parent, 0 for rows at or past n_nodes and for
// a parent outside [0, n_nodes).
template <int G>
__global__ void __launch_bounds__(128) validate_edges_kernel(const TreeDev a) {
    const Group<G> g;
    const int64_t total = a.nq * a.K, stride = (int64_t)gridDim.x * blockDim.x / G;
    for (int64_t e = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / G; e < total; e += stride) {
        const int64_t q = e / a.K;
        const int i = (int)(e - q * a.K), n = a.n_nodes[q];
        bool ok = false;
        if (i < n) {
            const int p = a.parent[e];
            if (p == -1) ok = true;
            else if (p >= 0 && p < n) {
                Grid m;
                if (map_grid(a.bits, a.n_maps, a.side, a.wpr, a.map_id ? a.map_id[q] : 0, m)) {
                    const double *uu = a.u + 5 * e;
                    ok = edge_free<G>(g, m, a.nx[q * a.K + p], a.ny[q * a.K + p], a.nx[e], a.ny[e], uu[0], uu[1], uu[2], uu[3]);
                }
            }
        }
        if (g.gl == 0) a.edge_ok[e] = ok ? 1 : 0;
    }
}

// The walks c_0 = i, c_1 = next(c_0), ... of every node i < n of one query at once, `steps` steps each, by pointer
// doubling over the whole CTA.  On entry T0[i] = next(i) * 2 | bit(i), with next(i) = -1 where a walk ends, and
// W[i] = i * 2 | 1.  Table T_k[i] packs (node 2^k steps from i, or -1 where the walk ends first) * 2 | AND of the bits
// of those 2^k nodes; T_{k+1} composes T_k with itself, and round k folds T_k into W when bit k of `steps` is set.  On
// exit W[i] = (node `steps` steps from i, or -1 where the walk ended first) * 2 | AND of the bits of the nodes it left.
// Exact whatever the order of the parents (they may point to higher indices) in ceil(log2(steps + 1)) rounds; the
// caller's barrier must separate the writes of T0 and W from the call.  K <= 2^30: an index and a bit share an int32.
__device__ __forceinline__ void chain_walk(int32_t *T0, int32_t *T1, int32_t *W, int n, int steps) {
    for (int k = 0; k < 31 && steps > 0 && (steps >> k) != 0; k++) {
        const int32_t *cur = (k & 1) ? T1 : T0;
        int32_t *nxt = (k & 1) ? T0 : T1;
        const bool take = (steps >> k) & 1, more = (steps >> (k + 1)) != 0;
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            if (take) {
                const int32_t s = W[i];
                const int pos = s >> 1;
                if (pos >= 0) {
                    TRRT_CHECK(pos < n);
                    const int32_t w = cur[pos];
                    W[i] = (w & ~1) | (s & w & 1);
                }
            }
            if (more) {
                int32_t w = cur[i];
                const int j = w >> 1;
                if (j >= 0) {
                    TRRT_CHECK(j < n);
                    const int32_t v = cur[j];
                    w = (v & ~1) | (w & v & 1);
                }
                nxt[i] = w;
            }
        }
        __syncthreads();
    }
}

// node_ok of one query per CTA: the AND of edge_ok over the nodes c_0 = i, c_1 = parent[c_0], ... of the walk
// main.path_nodes does, which follows parent for at most n_nodes - 1 steps and stops at a node without a parent (the
// cut of trrt_mission.cuh, so parent cycles through an overwritten root are well defined): chain_walk with next = parent
// and bit = edge_ok.
__global__ void __launch_bounds__(256) validate_chain_kernel(const TreeDev a) {
    const int K = a.K;
    for (int64_t q = blockIdx.x; q < a.nq; q += gridDim.x) {
        int32_t *T0 = a.work + q * 3 * (int64_t)K, *T1 = T0 + K, *W = T1 + K;
        const uint8_t *eok = a.edge_ok + q * (int64_t)K;
        uint8_t *nok = a.node_ok + q * (int64_t)K;
        const int n = min(max(a.n_nodes[q], 0), K);
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            const int p = a.parent[q * K + i];
            T0[i] = ((p >= 0 && p < n ? p : -1) * 2) | eok[i];
            W[i] = i * 2 | 1;
        }
        __syncthreads();
        chain_walk(T0, T1, W, n, n - 1);
        for (int i = threadIdx.x; i < K; i += blockDim.x) nok[i] = i < n ? (uint8_t)(W[i] & 1) : 0;
        __syncthreads();
        if (threadIdx.x == 0) {
            const int s = a.sol[q];
            a.sol_ok[q] = s < 0 ? (int8_t)-1 : (int8_t)(s < n ? nok[s] : 0);
        }
        __syncthreads(); // the next query of this CTA reuses nothing, but its tables start from a clean barrier
    }
}

// ---------------------------------------------------------------------------
// Tree repair
// ---------------------------------------------------------------------------
struct RepairDev {
    int64_t nq;
    int K;
    double *nx, *ny, *nth, *u;
    int32_t *parent, *n_nodes, *sol, *status;
    const int32_t *iters;
    const uint8_t *edge_ok;
    int32_t *new_index, *n_pruned;
    int32_t *work; // [nq][3][K]: the walk tables of chain_walk
};

constexpr int REPAIR_THREADS = 256;

// Exclusive prefix count of `flag` over the CTA, and the CTA's total.  Every thread of the CTA calls it.
__device__ __forceinline__ int block_count_before(bool flag, int &total, int *warp_count) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const unsigned b = __ballot_sync(0xffffffffu, flag);
    if (lane == 0) warp_count[wid] = __popc(b);
    __syncthreads();
    int before = __popc(b & ((1u << lane) - 1u));
    total = 0;
    for (int w = 0; w < REPAIR_THREADS / 32; w++) {
        const int c = warp_count[w];
        before += w < wid ? c : 0;
        total += c;
    }
    __syncthreads(); // warp_count is written again by the next call
    return before;
}

// One query per CTA.  Keep pass: chain_walk with node 0 absorbing (next(0) = 0, bit 1) and every other node stepping to
// its parent with bit edge_ok, or ending with bit 0 when its parent is outside [0, n) (-1 included): node i is kept
// when its walk of n - 1 steps stands at node 0 with every bit 1, i.e. it reaches node 0 within n - 1 parent steps over
// edges that edge_ok passes.  A kept node's parent walks a suffix of the same path, so the kept set is closed under
// parent.  Compaction: new_index is the exclusive count of kept rows before each row (-1 for pruned rows and rows >= n),
// in chunks of the CTA; then the rows move in place in increasing chunk order, each chunk read into registers before any
// of it is written (new <= old, so a chunk's writes land on rows already read), with parents remapped through the
// complete new_index.  The root leaves with parent -1 and u NaN, as rrt_setup plants it.
__global__ void __launch_bounds__(REPAIR_THREADS) repair_tree_kernel(const RepairDev a) {
    __shared__ int warp_count[REPAIR_THREADS / 32];
    const int K = a.K;
    for (int64_t q = blockIdx.x; q < a.nq; q += gridDim.x) {
        int32_t *T0 = a.work + q * 3 * (int64_t)K, *T1 = T0 + K, *W = T1 + K;
        const int64_t row0 = q * (int64_t)K;
        const uint8_t *eok = a.edge_ok + row0;
        int32_t *par = a.parent + row0, *nidx = a.new_index + row0;
        double *nx = a.nx + row0, *ny = a.ny + row0, *nth = a.nth + row0, *u = a.u + 5 * row0;
        const int n = min(max(a.n_nodes[q], 0), K);
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            const int p = par[i];
            T0[i] = i == 0 ? 1 : (p >= 0 && p < n && eok[i] ? p * 2 | 1 : -2);
            W[i] = i * 2 | 1;
        }
        __syncthreads();
        chain_walk(T0, T1, W, n, n - 1);
        int kept = 0;
        for (int base = 0; base < n; base += REPAIR_THREADS) { // new_index
            const int i = base + threadIdx.x;
            const bool keep = i < n && W[i] == 1;
            int total;
            const int before = block_count_before(keep, total, warp_count);
            if (i < n) nidx[i] = keep ? kept + before : -1;
            kept += total;
        }
        for (int i = n + threadIdx.x; i < K; i += blockDim.x) nidx[i] = -1;
        __syncthreads(); // new_index complete before any parent is remapped
        for (int base = 0; base < n; base += REPAIR_THREADS) { // rows, in place
            const int i = base + threadIdx.x;
            const int ni = i < n ? nidx[i] : -1;
            double x = 0, y = 0, th = 0, uu[5];
            int p = -1;
            if (ni >= 0) {
                TRRT_CHECK(ni <= i && ni < kept && (i == 0 || nidx[i - 1] < 0 || nidx[i - 1] == ni - 1));
                x = nx[i]; y = ny[i]; th = nth[i];
                if (i == 0) {
                    for (int j = 0; j < 5; j++) uu[j] = NAN;
                } else {
                    const int op = par[i];
                    TRRT_CHECK(op >= 0 && op < n && nidx[op] >= 0); // closure: a kept node's parent is kept
                    p = nidx[op];
                    for (int j = 0; j < 5; j++) uu[j] = u[5 * i + j];
                }
            }
            __syncthreads(); // the chunk is read before any of it is written
            if (ni >= 0) {
                nx[ni] = x; ny[ni] = y; nth[ni] = th; par[ni] = p;
                for (int j = 0; j < 5; j++) u[5 * ni + j] = uu[j];
            }
        }
        if (threadIdx.x == 0) {
            const int s = a.sol[q];
            const int ns = (s >= 0 && s < n) ? nidx[s] : -1;
            if (ns < 0 && a.status[q] == TRRT_OK_FOUND) a.status[q] = a.iters[q] < K - 1 ? TRRT_PAUSED : TRRT_OK_NOT_FOUND;
            a.sol[q] = ns;
            a.n_nodes[q] = kept;
            if (a.n_pruned) a.n_pruned[q] = n - kept;
        }
        __syncthreads(); // the next query of this CTA starts from a clean barrier
    }
}

// Race keys after a repair (the launcher fills them with 0xff first): min over the members that still hold
// TRRT_OK_FOUND of (iters << 32) | q, the key trrt_rrt_race_batch publishes.  Group ids outside [0, n_groups) race nobody.
__global__ void repair_race_kernel(const int32_t *__restrict__ status, const int32_t *__restrict__ iters,
                                   const int32_t *__restrict__ group, int64_t n_groups, unsigned long long *key, int64_t nq) {
    for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < nq; q += (int64_t)gridDim.x * blockDim.x) {
        const int g = group[q];
        if (status[q] == TRRT_OK_FOUND && g >= 0 && g < n_groups)
            atomicMin(key + g, ((unsigned long long)iters[q] << 32) | (unsigned long long)q);
    }
}

struct PathDev {
    const uint32_t *bits;
    int n_maps, side, wpr, mode, cap;
    const int32_t *map_id;
    int64_t n;
    const int32_t *route;  // mode 0: [n][cap][2]
    const double *rows;    // mode 1: [n][cap][8]
    const int32_t *row_seg; // mode 1: [n][cap]
    const int32_t *len, *status;
    uint8_t *step_ok, *ok;
};

// One warp per route or mission, G lanes per row.  mode 0 (Theta* routes): step 0 is search.freespace of the first
// waypoint, step t search.lineofsight(wp[t-1], wp[t]).  mode 1 (mission path rows): the edge test of row r-1 -> row r
// with row r's u when both rows belong to one segment, 1 at a segment's first row.  Rows past min(len, cap) are 0, and
// ok covers the stored rows only (steps past cap were not stored).
template <int G>
__global__ void __launch_bounds__(128) validate_path_kernel(const PathDev a) {
    const Group<G> g;
    const int lane = threadIdx.x & 31;
    const int64_t nw = (int64_t)gridDim.x * blockDim.x / 32;
    for (int64_t q = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / 32; q < a.n; q += nw) {
        const int len = min(max(a.len[q], 0), a.cap);
        Grid m;
        const bool map_ok = map_grid(a.bits, a.n_maps, a.side, a.wpr, a.map_id ? a.map_id[q] : 0, m);
        uint8_t *out = a.step_ok + q * (int64_t)a.cap;
        bool all = true;
        for (int r0 = 0; r0 < len; r0 += 32 / G) {
            const int r = r0 + lane / G;
            if (r >= len) continue; // group-uniform
            bool ok = map_ok;
            if (ok && a.mode == 0) {
                const int2 *wp = reinterpret_cast<const int2 *>(a.route) + q * (int64_t)a.cap;
                const int2 b = wp[r];
                if (r == 0) ok = m.freespace(b.x, b.y);
                else {
                    const int2 p = wp[r - 1];
                    ok = los_group<G>(g, m, p.x, p.y, b.x, b.y);
                }
            } else if (ok && r > 0 && a.row_seg[q * a.cap + r] == a.row_seg[q * a.cap + r - 1]) {
                const double *b = a.rows + (q * a.cap + r) * 8, *p = b - 8;
                ok = edge_free<G>(g, m, p[0], p[1], b[0], b[1], b[3], b[4], b[5], b[6]);
            }
            if (g.gl == 0) out[r] = ok ? 1 : 0;
            all = all && ok;
        }
        all = __all_sync(0xffffffffu, all);
        for (int r = len + lane; r < a.cap; r += 32) out[r] = 0;
        if (lane == 0) a.ok[q] = (a.status[q] == 0 && all) ? 1 : 0;
    }
}

} // namespace trrt
