// trrt_mission.cuh -- batched main.py missions (main.py:56-84): per mission, a chain of RRT segments between
// consecutive waypoints, restarting from the rrt.findnearest node once a segment has failed.
//
// A mission's chain is kept on the device.  trrt_mission_batch runs, per stage s (segment s of every mission that has
// one), three launches on the caller's stream:
//   mission_stage_kernel   start / goal rows and the K-1 rand_conf samples of segment s, in the layout of trrt_rrt_batch
//   trrt_rrt_batch         the fused RRT kernel (trrt_rrt.cuh), unchanged, over the first n_active[s] slots
//   mission_commit_kernel  segment records, rrt.findnearest for failed segments, path rows, next mission state
// Missions are dispatched in decreasing number of segments (d_order: slot -> mission), so the missions with a segment
// s are exactly the first n_active[s] slots and no compaction is needed between stages.
#pragma once
#include "trrt_bike.cuh"
#include "trrt_rng.cuh"

namespace trrt {

// rrt.findnearest (rrt.py:117-128) over the edge log of one tree, by one block of FN_THREADS threads.  The reference
// walks parents in tree order and children in append order with a strict `<`, i.e. it returns the edge minimising
// (distance, parent index, iteration) lexicographically.  nx/ny/nth [K], it_near/it_new [K-1] of that tree.
// Every thread receives best (node index, -1 when the tree has no child entry) and its distance.
constexpr int FN_THREADS = 128;
__device__ __forceinline__ void findnearest_block(const BikeParams &P, int K, const double *__restrict__ nx, const double *__restrict__ ny,
                                                  const double *__restrict__ nth, const int32_t *__restrict__ it_near,
                                                  const int32_t *__restrict__ it_new, double gx, double gy, double gth, int &best,
                                                  double &best_dist) {
    double bd = INFINITY;
    int bp = 0x7fffffff, bit = 0x7fffffff, bc = -1;
    for (int it = threadIdx.x; it < K - 1; it += FN_THREADS) {
        int c = it_new[it];
        if (c < 0) continue;
        int p = it_near[it];
        double dx = gx - nx[c], dy = gy - ny[c];
        double d = P.weightxy * sqrt(dx * dx + dy * dy) + (1 - P.weightxy) * fabs(anglediff(nth[c], gth));
        if (d < bd || (d == bd && (p < bp || (p == bp && it < bit)))) { bd = d; bp = p; bit = it; bc = c; }
    }
    __shared__ double sd[FN_THREADS];
    __shared__ int sp[FN_THREADS], si[FN_THREADS], sc[FN_THREADS];
    sd[threadIdx.x] = bd; sp[threadIdx.x] = bp; si[threadIdx.x] = bit; sc[threadIdx.x] = bc;
    __syncthreads();
    for (int off = FN_THREADS / 2; off > 0; off >>= 1) {
        if ((int)threadIdx.x < off) {
            int o = threadIdx.x + off;
            if (sc[o] >= 0 && (sc[threadIdx.x] < 0 || sd[o] < sd[threadIdx.x] ||
                               (sd[o] == sd[threadIdx.x] && (sp[o] < sp[threadIdx.x] || (sp[o] == sp[threadIdx.x] && si[o] < si[threadIdx.x]))))) {
                sd[threadIdx.x] = sd[o]; sp[threadIdx.x] = sp[o]; si[threadIdx.x] = si[o]; sc[threadIdx.x] = sc[o];
            }
        }
        __syncthreads();
    }
    best = sc[0];
    best_dist = sc[0] >= 0 ? sd[0] : NAN;
    __syncthreads(); // the shared arrays may be reused by the caller's next call
}

// status of a mission whose chain stopped because rrt.findnearest found no node (main.py:79-81 raises TypeError);
// kept in step with trrt_status in thetarrt.h
constexpr int MISSION_NO_NEAREST = 7;
constexpr int SEG_NOT_RUN = 255;
constexpr int MISSION_THREADS = 128;

struct MissionDev {
    int H, W;
    const int32_t *map_id; // [n] or null
    BikeParams P;
    double xystdv, anglestdv;
    int64_t n;
    int K;
    const int32_t *wp; // [n][wp_cap][2]
    int wp_cap;
    const int32_t *n_wp, *route_status;
    const double *normals;
    const int64_t *nrange; // [n][2]
    const int32_t *order;  // slot -> mission
    // outputs
    int seg_cap;
    double *seg_begin, *seg_end, *seg_solution, *seg_nearest, *seg_mindist;
    int32_t *seg_n_nodes, *seg_n_edges, *seg_iters, *seg_status;
    int32_t *status, *stop_seg, *n_seg;
    double *path;
    int32_t *path_seg;
    int path_cap;
    int32_t *path_len;
    // per-mission state (workspace)
    int64_t *off;    // next unread normal
    double *restart; // [n][3] most recent findnearest node
    int32_t *restarted;
    // per-slot rows of the running stage (workspace), read and written by trrt_rrt_batch
    double *q_start, *q_goal;
    int32_t *q_map, *q_sxy;
    double *q_sth;
    double *nx, *ny, *nth, *u;
    int32_t *parent, *q_n_nodes, *q_sol, *q_status, *q_iters, *it_near, *it_new;
};

// Every mission: its segment count, its outputs cleared, its state at the start of the chain.  A route that is not
// TRRT_OK_FOUND is copied with zero segments (main.plan returns False, or the reference raises, before any RRT).
__global__ void __launch_bounds__(MISSION_THREADS) mission_init_kernel(const MissionDev a) {
    for (int64_t m = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; m < a.n; m += (int64_t)gridDim.x * blockDim.x) {
        const int rs = a.route_status ? a.route_status[m] : TRRT_OK_FOUND;
        const int nw = a.n_wp[m];
        int st = rs, ns = 0;
        if (rs == TRRT_OK_FOUND) {
            if (nw > a.wp_cap || nw - 1 > a.seg_cap) st = TRRT_ERR_CAPACITY;
            else ns = nw > 1 ? nw - 1 : 0;
        }
        a.status[m] = st;
        a.stop_seg[m] = st == TRRT_OK_FOUND ? -1 : 0;
        a.n_seg[m] = ns;
        a.path_len[m] = 0;
        a.off[m] = a.nrange[2 * m];
        a.restarted[m] = 0;
        for (int s = 0; s < a.seg_cap; s++) {
            const int64_t r = m * a.seg_cap + s;
            for (int j = 0; j < 3; j++) {
                a.seg_begin[3 * r + j] = NAN; a.seg_end[3 * r + j] = NAN; a.seg_solution[3 * r + j] = NAN; a.seg_nearest[3 * r + j] = NAN;
            }
            a.seg_mindist[r] = NAN;
            a.seg_n_nodes[r] = 0; a.seg_n_edges[r] = 0; a.seg_iters[r] = 0;
            a.seg_status[r] = SEG_NOT_RUN;
        }
    }
}

// main.py:58-68 for segment s of the mission in slot blockIdx.x: headings, restart point, and the rand_conf stream of
// rrt.rrt drawn around the segment's end (samples.stream_from_normals: fp64, no contraction, clip, truncate,
// standardangle).  A slot whose mission has stopped gets a query that rejects every sample at once (samples equal to
// the start node), so the RRT launch spends next to nothing on it and the commit ignores it.
__global__ void __launch_bounds__(MISSION_THREADS) mission_stage_kernel(const MissionDev a, int s) {
    const int64_t slot = blockIdx.x;
    const int64_t m = a.order[slot];
    const int K = a.K;
    __shared__ double row[6]; // begin x, y, theta, end x, y, theta
    __shared__ int64_t off;
    __shared__ int live;
    if (threadIdx.x == 0) {
        int lv = a.status[m] == TRRT_OK_FOUND && s < a.n_seg[m];
        double b0 = 0, b1 = 0, b2 = 0, e0 = 0, e1 = 0, e2 = 0;
        if (lv && a.off[m] + 3 * (int64_t)(K - 1) > a.nrange[2 * m + 1]) { // too few normals for this segment
            a.status[m] = TRRT_ERR_CAPACITY;
            a.stop_seg[m] = s;
            lv = 0;
        }
        if (lv) {
            const int32_t *w = a.wp + m * (int64_t)a.wp_cap * 2;
            const int x0 = w[2 * s], y0 = w[2 * s + 1], x1 = w[2 * s + 2], y1 = w[2 * s + 3];
            double angle1 = anglebetween(1, 0, (double)(x1 - x0), (double)(y1 - y0)); // main.py:59
            b0 = x0; b1 = y0;
            if (a.restarted[m]) { // main.py:60-62: every segment after a failed one starts at the nearest node
                b0 = a.restart[3 * m]; b1 = a.restart[3 * m + 1]; angle1 = a.restart[3 * m + 2];
            }
            double angle2 = angle1; // main.py:63-64: last segment
            if (s + 2 < a.n_wp[m]) angle2 = anglebetween(1, 0, (double)(w[2 * s + 4] - x1), (double)(w[2 * s + 5] - y1));
            b2 = standardangle(angle1);
            e0 = x1; e1 = y1; e2 = standardangle(angle2);
            double *ob = a.seg_begin + 3 * (m * a.seg_cap + s), *oe = a.seg_end + 3 * (m * a.seg_cap + s);
            ob[0] = b0; ob[1] = b1; ob[2] = b2; oe[0] = e0; oe[1] = e1; oe[2] = e2;
        }
        row[0] = b0; row[1] = b1; row[2] = b2; row[3] = e0; row[4] = e1; row[5] = e2;
        a.q_start[3 * slot] = b0; a.q_start[3 * slot + 1] = b1; a.q_start[3 * slot + 2] = b2;
        a.q_goal[3 * slot] = e0; a.q_goal[3 * slot + 1] = e1; a.q_goal[3 * slot + 2] = e2;
        if (a.map_id) a.q_map[slot] = a.map_id[m];
        off = a.off[m];
        live = lv;
    }
    __syncthreads();
    int32_t *sxy = a.q_sxy + slot * (int64_t)(K - 1) * 2;
    double *sth = a.q_sth + slot * (int64_t)(K - 1);
    if (!live) {
        for (int j = threadIdx.x; j < K - 1; j += blockDim.x) { sxy[2 * j] = 0; sxy[2 * j + 1] = 0; sth[j] = 0.0; }
        return;
    }
    const double gx = row[3], gy = row[4], gth = standardangle(row[5]);
    const double sx = a.xystdv * (double)a.H, sy = a.xystdv * (double)a.W, hm = (double)(a.H - 1), wm = (double)(a.W - 1);
    const double *z = a.normals + off;
    for (int j = threadIdx.x; j < K - 1; j += blockDim.x)
        rand_conf_sample(z + 3 * j, gx, gy, gth, sx, sy, hm, wm, a.anglestdv, sxy[2 * j], sxy[2 * j + 1], sth[j]);
}

// main.py:68-79 after rrt.rrt returned, for the mission in slot blockIdx.x: the segment record, rrt.findnearest when
// the segment failed, the path rows of main.path_nodes (root .. solution or nearest node, by walking `parent`), and
// the mission state of the next segment.
__global__ void __launch_bounds__(MISSION_THREADS) mission_commit_kernel(const MissionDev a, int s) {
    const int64_t slot = blockIdx.x;
    const int64_t m = a.order[slot];
    const int K = a.K;
    __shared__ int live, n_edges;
    if (threadIdx.x == 0) {
        live = a.status[m] == TRRT_OK_FOUND && s < a.n_seg[m];
        n_edges = 0;
    }
    __syncthreads();
    if (!live) return;
    const int32_t *it_near = a.it_near + slot * (int64_t)(K - 1), *it_new = a.it_new + slot * (int64_t)(K - 1);
    const double *nx = a.nx + slot * (int64_t)K, *ny = a.ny + slot * (int64_t)K, *nth = a.nth + slot * (int64_t)K;
    int cnt = 0;
    for (int it = threadIdx.x; it < K - 1; it += blockDim.x) cnt += it_new[it] >= 0;
    atomicAdd(&n_edges, cnt);
    const int rs = a.q_status[slot], sol = a.q_sol[slot];
    const bool ok = rs == TRRT_OK_FOUND || rs == TRRT_OK_NOT_FOUND;
    int best = -1;
    double best_dist = NAN;
    if (ok && sol < 0) // rrt.findnearest(graph, end) (main.py:73)
        findnearest_block(a.P, K, nx, ny, nth, it_near, it_new, a.q_goal[3 * slot], a.q_goal[3 * slot + 1], a.q_goal[3 * slot + 2], best,
                          best_dist);
    __syncthreads();
    if (threadIdx.x != 0) return;
    const int64_t r = m * a.seg_cap + s;
    const int nn = a.q_n_nodes[slot], iters = a.q_iters[slot];
    a.seg_n_nodes[r] = nn;
    a.seg_n_edges[r] = n_edges;
    a.seg_iters[r] = iters;
    a.seg_status[r] = rs;
    if (!ok) { a.status[m] = rs; a.stop_seg[m] = s; return; } // rrt.rrt raises (TRRT_ERR_REF_RAISES_DRIVE_NONE)
    if (sol >= 0) {
        a.seg_solution[3 * r] = nx[sol]; a.seg_solution[3 * r + 1] = ny[sol]; a.seg_solution[3 * r + 2] = nth[sol];
    } else if (best >= 0) {
        a.seg_nearest[3 * r] = nx[best]; a.seg_nearest[3 * r + 1] = ny[best]; a.seg_nearest[3 * r + 2] = nth[best];
        a.seg_mindist[r] = best_dist;
        a.restart[3 * m] = nx[best]; a.restart[3 * m + 1] = ny[best]; a.restart[3 * m + 2] = nth[best];
        a.restarted[m] = 1;
    } else { a.status[m] = MISSION_NO_NEAREST; a.stop_seg[m] = s; return; } // main.py:79-81: TypeError
    // main.path_nodes: terminal node back to the root through cameFrom, stored root first.  A walk longer than the tree
    // (the root's cameFrom entry overwritten by a later edge, rrt.py:187-188) is cut at n_nodes rows.
    const int32_t *par = a.parent + slot * (int64_t)K;
    const double *u = a.u + slot * (int64_t)K * 5;
    const int term = sol >= 0 ? sol : best;
    int len = 0;
    for (int c = term; c >= 0 && len < nn; c = par[c]) len++;
    const int base = a.path_len[m];
    int c = term;
    for (int k = len - 1; k >= 0; k--, c = par[c]) {
        const int64_t row = (int64_t)base + k;
        if (row >= a.path_cap) continue;
        double *o = a.path + (m * a.path_cap + row) * 8;
        o[0] = nx[c]; o[1] = ny[c]; o[2] = nth[c];
        for (int j = 0; j < 5; j++) o[3 + j] = u[5 * c + j];
        a.path_seg[m * a.path_cap + row] = s;
    }
    a.path_len[m] = base + len;
    a.off[m] += 3 * (int64_t)iters; // rrt.rrt draws one sample per iteration it runs (rrt.py:144, stops at its break)
}

} // namespace trrt
