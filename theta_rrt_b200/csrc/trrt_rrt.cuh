// trrt_rrt.cuh -- K2: the fused rrt.rrt loop (rrt.py:130-206), G lanes per query.
//
// Two schedules produce bit-identical results:
//
//  * cooperative (schedule 1): the G lanes of a group work on ONE loop iteration at a time: the
//    nearest scan, the Bresenham rays and the circle raster are lane-parallel, the scalar steer /
//    drive math is computed redundantly by every lane.
//
//  * speculative window (schedule 0, default): the sample stream does not depend on the tree
//    (rrt.py:144 draws before any test), and everything an iteration does after picking its
//    nearest node depends only on (nearest node, sample, map).  So lane j of a group expands
//    iteration k0+j against a SNAPSHOT of the tree: nearest scan (pooled over the warps of the CTA
//    and staged through shared memory), steer, clearance rays, re-drive and edge raster.  The
//    nodes the window would insert are then folded forward in iteration order (registers and
//    shuffles): later lanes learn whether one of them is strictly nearer than their snapshot winner
//    (new nodes have higher indices, so the snapshot winner keeps ties) and whether it equals their
//    sample or their new node.  The window commits, in parallel, all lanes before the first one
//    whose nearest node was inserted in this very window (24.6 of 32 on cfg 3), and the next window
//    starts at that iteration.  The committed sequence is exactly the sequential loop.  One
//    persistent kernel, groups pull queries from a counter.
#pragma once
#include "trrt_bike.cuh"
#include "trrt_lane.cuh"

namespace trrt {

struct RrtDev {
    const uint32_t *bits;
    int H, W, wpr;
    const int32_t *map_id;
    BikeParams P;
    int64_t nq;
    int K;
    const double *start, *goal;
    const int32_t *sxy; // int32 pairs, or int16 pairs when sxy16 is set
    int sxy16;
    const double *sth;
    double *nx, *ny, *nth;
    int32_t *parent;
    double *u;
    int32_t *n_nodes, *sol, *status, *iters;
    int32_t *it_near, *it_new;
    uint8_t *it_code, *los_log;
    int32_t *n_los;
    unsigned long long *counters;
    int32_t *tab; // [nq][tsize] open-addressing index table for the `in G.keys()` tests
    int tsize;
    unsigned long long *next_query; // work counter of the persistent speculative kernel (zeroed by the launcher)
    // optional packed copy of the rows that exist (see trrt_rrt_args in thetarrt.h)
    unsigned long long *pack_rows;
    long long *row_start;
    double *px, *py, *pth, *pu;
    int32_t *pparent;
    // pause and resume (see trrt_rrt_args in thetarrt.h): per-query stop iteration or nullptr (K-1); resume paused queries
    const int32_t *stop_at;
    int resume;
    // seed races (see trrt_rrt_race in thetarrt.h): race group of each query or nullptr (no race), and per group the
    // key (iters << 32) | q of the best FOUND member published so far, ~0 = none
    const int32_t *race_group;
    int64_t n_race_groups;
    unsigned long long *race_key;
};

__device__ __forceinline__ unsigned hash3(double x, double y, double t) {
    // value-equality hash: -0.0 and +0.0 must collide (Python: -0.0 == 0.0)
    unsigned long long a = (unsigned long long)__double_as_longlong(x + 0.0);
    unsigned long long b = (unsigned long long)__double_as_longlong(y + 0.0);
    unsigned long long c = (unsigned long long)__double_as_longlong(t + 0.0);
    unsigned long long h = a * 0x9E3779B97F4A7C15ull;
    h ^= (b + 0x7F4A7C159E3779B9ull + (h << 6) + (h >> 2));
    h *= 0xC2B2AE3D27D4EB4Full;
    h ^= (c + 0x165667B19E3779F9ull + (h << 6) + (h >> 2));
    h ^= h >> 29;
    h *= 0x94D049BB133111EBull;
    h ^= h >> 32;
    return (unsigned)h;
}

// index of the tree node equal (by value) to (x, y, t), or -1   [rrt.py:151, :179]
__device__ __noinline__ int tree_find(const int32_t *tab, int tmask, const double *nx, const double *ny, const double *nth, double x,
                                         double y, double t, unsigned long long &probes) {
    unsigned s = hash3(x, y, t) & (unsigned)tmask;
    for (;;) {
        int e = tab[s];
        probes++;
        if (e == 0) return -1;
        int i = e - 1;
        if (nx[i] == x && ny[i] == y && nth[i] == t) return i;
        s = (s + 1) & (unsigned)tmask;
    }
}
__device__ __noinline__ void tree_insert(int32_t *tab, int tmask, double x, double y, double t, int idx) {
    unsigned s = hash3(x, y, t) & (unsigned)tmask;
    while (tab[s] != 0) s = (s + 1) & (unsigned)tmask;
    tab[s] = idx + 1;
}
// tree_find that also reports where its probe sequence ended: for a miss that is the first empty slot on the key's
// probe path.  Nothing is ever deleted, so an insert of the same key may resume there instead of hashing again
// (the commit loop is a serial chain: every instruction and every dependent load taken out of it counts --
// 69.6 -> 66.2 ms per cfg-3 step).  Inlined (one call site): as a call, its probe counter and slot were on the caller's stack
// (cfg 3: 28.94 ms inlined, 29.78 ms as a call; profiles/r6/NOTES.md).
__device__ __forceinline__ int tree_find_slot(const int32_t *tab, int tmask, const double *nx, const double *ny, const double *nth, double x,
                                              double y, double t, unsigned long long &probes, int &slot) {
    unsigned s = hash3(x, y, t) & (unsigned)tmask;
    for (;;) {
        int e = tab[s];
        probes++;
        if (e == 0) { slot = (int)s; return -1; }
        int i = e - 1;
        if (nx[i] == x && ny[i] == y && nth[i] == t) { slot = (int)s; return i; }
        s = (s + 1) & (unsigned)tmask;
    }
}
__device__ __forceinline__ void tree_insert_from(int32_t *tab, int tmask, int slot, int idx) {
    unsigned s = (unsigned)slot;
    while (tab[s] != 0) s = (s + 1) & (unsigned)tmask; // slots taken since the lookup
    tab[s] = idx + 1;
}

// the same for lanes of one warp inserting different keys at the same time (parallel segment commit)
__device__ __forceinline__ void tree_insert_cas(int32_t *tab, int tmask, int slot, int idx) {
    unsigned s = (unsigned)slot;
    TRRT_CHECK(slot >= 0 && slot <= tmask);
    while (atomicCAS(tab + s, 0, idx + 1) != 0) s = (s + 1) & (unsigned)tmask;
}

// Outcome of one iteration from "nearest node chosen" to "edge tested" (rrt.py:161-176).
enum { EX_ACCEPT = 100 }; // edge is free: proceed to insert (rrt.py:179)
struct Expand {
    double wx, wy, wth;                  // qnew (after the optional 1/3 re-drive)
    double usteer, iccx, iccy, rad, udist; // u as stored in cameFrom
    int code;                            // TRRT_IT_STEER_CONSTRAINT / TRRT_IT_ARC_BLOCKED / EX_ACCEPT
    int flags;                           // bit0 straight, bit1 reference raises (Q7), bit2 goal reached,
                                         // bits 4-5 number of LOS calls, bit 6/7 their results
    int lospx, arcpx, arcang;            // counters of this iteration
    int drive;
};

// Everything after the nearest node is known.  GA lanes share the rays / raster; GA == 1 is one lane working
// alone (speculative schedule) and takes the single-lane code of trrt_lane.cuh.
template <int GA>
__device__ __forceinline__ bool ray_clear(const Group<GA> &ga, const Grid &m, long long ax, long long ay, long long bx, long long by, int *px) {
    if (GA == 1) { *px += los_lane_pixels(m, ax, ay, bx, by); return los_lane(m, ax, ay, bx, by); }
    unsigned long long p = 0;
    bool ok = los_group<GA>(ga, m, ax, ay, bx, by, &p);
    *px += (int)p;
    return ok;
}

// Inlined: one call site per kernel; measured on cfg 3: inlined 38.8 ms, as a call 39.4 ms.
template <int GA>
__device__ __forceinline__ void expand_from(const Group<GA> &ga, const Grid &m, const BikeParams &P, double ox, double oy, double oth,
                                           double qx, double qy, double qth, double gx, double gy, double gth, Expand &e_out) {
    // results are built in locals (only the inlined ray_clear takes the address of a pixel counter; no call receives a
    // reference or a pointer), so that after inlining the caller's Expand stays in registers
    Expand e;
    int lospx = 0, arcpx = 0, arcang = 0;
    Steer s;
    steer(P, ox, oy, oth, qx, qy, qth, s);
    e.wx = s.x; e.wy = s.y; e.wth = s.theta;
    e.usteer = s.steer; e.iccx = s.iccx; e.iccy = s.iccy; e.rad = s.rad; e.udist = s.dist;
    e.flags = s.straight ? 1 : 0;
    e.lospx = e.arcpx = e.arcang = e.drive = 0;
    double us = standardangle(s.steer);
    if (us < P.leftconstraint || us > P.rightconstraint) { e.code = TRRT_IT_STEER_CONSTRAINT; e_out = e; return; } // rrt.py:166
    // clearance (rrt.py:169): valid, bike_clear, front_of_bike_clear with short-circuit
    int nlos = 0;
    bool ok = m.inb(trunc_ll(e.wx), trunc_ll(e.wy));
    if (ok) {
        const Rot Rw = rot_make(e.wth); // bike_clear and front_of_bike_clear rotate by the same heading (rrt.py:210,217)
        double bx, by;
        rot_apply(Rw, P.bikelength, 0.0, bx, by);
        ok = ray_clear<GA>(ga, m, trunc_ll(e.wx), trunc_ll(e.wy), trunc_ll(bx + e.wx), trunc_ll(by + e.wy), &lospx);
        if (ok) e.flags |= 1 << 6;
        nlos = 1;
        if (ok) {
            rot_apply(Rw, P.bikelength * P.frontclearance, 0.0, bx, by);
            ok = ray_clear<GA>(ga, m, trunc_ll(e.wx), trunc_ll(e.wy), trunc_ll(bx + e.wx), trunc_ll(by + e.wy), &lospx);
            if (ok) e.flags |= 1 << 7;
            nlos = 2;
        }
    }
    e.flags |= nlos << 4;
    if (!ok) {
        if (s.straight) { e.flags |= 2; e.code = TRRT_IT_NOT_RUN; e.lospx = lospx; e_out = e; return; } // rrt.py:170-171 -> TypeError in the reference
        e.udist = s.dist / 3;
        const Pose d = drive_bf(P, ox, oy, s.bfx, s.bfy, s.steer, s.iccx, s.iccy, s.rad, e.udist);
        e.wx = d.x; e.wy = d.y; e.wth = d.theta;
        e.drive = 1;
    }
    // goal test input (rrt.py:191-198) depends only on qnew
    {
        double dgx = gx - e.wx, dgy = gy - e.wy;
        if (sqrt(dgx * dgx + dgy * dgy) < P.tol_xy && fabs(anglediff(e.wth, gth)) < P.tol_ang) e.flags |= 4;
    }
    // edge collision (rrt.py:173-176)
    bool blocked;
    if (s.straight) {
        blocked = !ray_clear<GA>(ga, m, trunc_ll(ox), trunc_ll(oy), trunc_ll(e.wx), trunc_ll(e.wy), &arcpx);
    } else if (GA == 1) {
        const ArcLane r = arc_blocked_lane(m, ox, oy, e.wx, e.wy, s.steer, s.iccx, s.iccy, s.rad);
        blocked = r.blocked; arcpx = r.cand_px; arcang = r.angle_tests;
    } else {
        unsigned long long apx = 0, aang = 0;
        blocked = arc_blocked<GA>(ga, m, ox, oy, e.wx, e.wy, s.steer, s.iccx, s.iccy, s.rad, &apx, &aang);
        apx = ga.sum(apx); aang = ga.sum(aang);
        arcpx = (int)apx; arcang = (int)aang;
    }
    e.code = blocked ? TRRT_IT_ARC_BLOCKED : EX_ACCEPT;
    e.lospx = lospx; e.arcpx = arcpx; e.arcang = arcang;
    e_out = e;
}

// fp64 nearest scan over nodes [0, n), G lanes cooperating (strided); result in every lane  (rrt.py:156-158)
template <int G>
__device__ __forceinline__ int nearest_coop(const Group<G> &g, const double *nx, const double *ny, int n, double qx, double qy) {
    double bd = INFINITY;
    int bi = 0x7fffffff;
    int i = g.gl;
    for (; i + 3 * G < n; i += 4 * G) {
        double x0 = nx[i], y0 = ny[i], x1 = nx[i + G], y1 = ny[i + G];
        double x2 = nx[i + 2 * G], y2 = ny[i + 2 * G], x3 = nx[i + 3 * G], y3 = ny[i + 3 * G];
        double dx, dy, d;
        dx = qx - x0; dy = qy - y0; d = dx * dx + dy * dy; if (d < bd) { bd = d; bi = i; }
        dx = qx - x1; dy = qy - y1; d = dx * dx + dy * dy; if (d < bd) { bd = d; bi = i + G; }
        dx = qx - x2; dy = qy - y2; d = dx * dx + dy * dy; if (d < bd) { bd = d; bi = i + 2 * G; }
        dx = qx - x3; dy = qy - y3; d = dx * dx + dy * dy; if (d < bd) { bd = d; bi = i + 3 * G; }
    }
    for (; i < n; i += G) {
        double dx = qx - nx[i], dy = qy - ny[i];
        double d = dx * dx + dy * dy;
        if (d < bd) { bd = d; bi = i; }
    }
    g.min_di(bd, bi);
    return bi;
}

struct RrtQuery {
    Grid m;
    double *nx, *ny, *nth;
    int32_t *parent;
    double *uo;
    const int32_t *sxy;
    const double *sth;
    int32_t *it_near, *it_new;
    uint8_t *it_code, *los_log;
    int32_t *tab;
    int tmask;
    int limit; // iterations it < limit run (d_stop_at clamped to [0, K-1]); fits the padding after tmask
    double gx, gy, gth;
};
// one copy per warp of rrt_kernel_spec<32> sits in its static shared memory, which has 184 bytes to spare
static_assert(sizeof(RrtQuery) == 152, "RrtQuery grew: rrt_kernel_spec's shared memory budget");

// the query's stop: iterations it < limit run
__device__ __forceinline__ int query_limit(const RrtDev &a, int64_t q) {
    if (!a.stop_at) return a.K - 1;
    const int s = a.stop_at[q];
    return s < 0 ? 0 : (s > a.K - 1 ? a.K - 1 : s);
}

// Seed races.  A member of race group g runs no iteration it >= best[g], the smallest iters of a member of g that ended
// with TRRT_OK_FOUND.  Members publish with atomicMin on race_key[g] = (iters << 32) | q, so the key keeps the lowest
// query index among equal iteration counts.  A member reads the key while it runs: a stale value is >= the final best[g]
// and only delays a cut, so the members that solve at best[g] are never cut and the winner does not depend on timing.
// Group ids outside [0, n_race_groups) race nobody.
__device__ __forceinline__ int race_group_of(const RrtDev &a, int64_t q) {
    const int gi = a.race_group[q];
    return (gi >= 0 && gi < a.n_race_groups) ? gi : -1;
}
__device__ __forceinline__ unsigned long long race_key_load(const unsigned long long *p) {
    unsigned long long v; // bypasses L1: other SMs publish into L2
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p));
    return v;
}
// lim lowered to the best[g] the group's key shows now (a.race_group set; one lane reads, the caller broadcasts)
__device__ __forceinline__ int race_limit(const RrtDev &a, int64_t q, int lim) {
    const int gi = race_group_of(a, q);
    if (gi < 0) return lim;
    TRRT_CHECK(gi < a.n_race_groups);
    const unsigned long long best = race_key_load(a.race_key + gi) >> 32; // 0xffffffff: no member has found the goal
    return best < (unsigned long long)lim ? (int)best : lim;
}
// the same bound, read by the group's leader and the same in every lane
template <int G>
__device__ __forceinline__ int race_limit_group(const RrtDev &a, int64_t q, const Group<G> &g, int lim) {
    if (!a.race_group) return lim;
    return g.bcast(g.gl == 0 ? race_limit(a, q, lim) : lim, 0);
}

// a resume call continues query q: it is paused and its stop (and its race group's best) lies beyond the iterations it
// has run
template <int G>
__device__ __forceinline__ bool query_resumes(const RrtDev &a, int64_t q, const Group<G> &g) {
    return a.status[q] == TRRT_PAUSED && a.iters[q] < race_limit_group<G>(a, q, g, query_limit(a, q));
}

// pointers of query q (no memory is touched)
__device__ __forceinline__ void rrt_ptrs(const RrtDev &a, int64_t q, RrtQuery &Q) {
    const int K = a.K;
    Q.m.W = a.W; Q.m.H = a.H; Q.m.wpr = a.wpr;
    Q.m.bits = a.bits + (a.map_id ? (size_t)a.map_id[q] * a.H * a.wpr : 0);
    Q.nx = a.nx + q * K; Q.ny = a.ny + q * K; Q.nth = a.nth + q * K;
    Q.parent = a.parent + q * K;
    Q.uo = a.u ? a.u + q * (int64_t)K * 5 : nullptr;
    Q.sxy = a.sxy + q * (int64_t)(K - 1) * (a.sxy16 ? 1 : 2);
    Q.sth = a.sth + q * (int64_t)(K - 1);
    Q.it_near = a.it_near ? a.it_near + q * (int64_t)(K - 1) : nullptr;
    Q.it_new = a.it_new ? a.it_new + q * (int64_t)(K - 1) : nullptr;
    Q.it_code = a.it_code ? a.it_code + q * (int64_t)(K - 1) : nullptr;
    Q.los_log = a.los_log ? a.los_log + q * (int64_t)(K - 1) * 2 : nullptr;
    Q.tab = a.tab + q * (int64_t)a.tsize;
    Q.tmask = a.tsize - 1;
    Q.limit = query_limit(a, q);
    Q.gx = a.goal[3 * q]; Q.gy = a.goal[3 * q + 1]; Q.gth = standardangle(a.goal[3 * q + 2]);
}

// rand_conf's (x, y) of iteration `it` (rrt.py:144): int32 pairs, or int16 pairs (half the host-to-device bytes)
__device__ __forceinline__ void sample_xy(const RrtDev &a, const RrtQuery &Q, int it, int &sx, int &sy) {
    if (a.sxy16) {
        const short2 v = __ldg(reinterpret_cast<const short2 *>(Q.sxy) + it);
        sx = v.x; sy = v.y;
    } else {
        const int2 v = __ldg(reinterpret_cast<const int2 *>(Q.sxy) + it);
        sx = v.x; sy = v.y;
    }
}

// pointers + empty index + the start node (rrt.py:132-138)
template <int G>
__device__ __forceinline__ void rrt_setup(const RrtDev &a, int64_t q, const Group<G> &g, RrtQuery &Q) {
    rrt_ptrs(a, q, Q);
#pragma unroll 4
    for (int i = g.gl; i < a.tsize; i += G) Q.tab[i] = 0;
    if (g.gl == 0) {
        Q.nx[0] = a.start[3 * q]; Q.ny[0] = a.start[3 * q + 1]; Q.nth[0] = standardangle(a.start[3 * q + 2]);
        Q.parent[0] = -1;
        if (Q.uo) for (int j = 0; j < 5; j++) Q.uo[j] = NAN;
    }
    g.sync();
    if (g.gl == 0) tree_insert(Q.tab, Q.tmask, Q.nx[0], Q.ny[0], Q.nth[0], 0);
    g.sync();
}

// A paused query (resume calls): pointers, the loop state left in the output arrays, and its index rebuilt over nodes
// [0, n) by the group.  The nodes are distinct keys, so every insertion order gives a table with the same lookups (only
// the probe counts differ).  Node 0 and the counter row are not touched.
template <int G>
__device__ __forceinline__ void rrt_setup_resume(const RrtDev &a, int64_t q, const Group<G> &g, RrtQuery &Q, int &n, int &iters,
                                                 int &nlos) {
    rrt_ptrs(a, q, Q);
    n = a.n_nodes[q];
    iters = a.iters[q];
    nlos = a.n_los ? a.n_los[q] : 0;
    TRRT_CHECK(n >= 1 && n <= a.K && iters >= 0 && iters < Q.limit);
#pragma unroll 4
    for (int i = g.gl; i < a.tsize; i += G) Q.tab[i] = 0;
    g.sync();
    for (int i = g.gl; i < n; i += G) {
        const double x = Q.nx[i], y = Q.ny[i], t = Q.nth[i];
        tree_insert_cas(Q.tab, Q.tmask, (int)(hash3(x, y, t) & (unsigned)Q.tmask), i);
    }
    g.sync();
}

// rrt.py:179-201 for an accepted edge.  Uniform across the group; the leader writes.  Returns the node index.
template <int G>
__device__ __forceinline__ int rrt_insert(const Group<G> &g, const RrtQuery &Q, const Expand &e, int near, int K, int &n, int &code,
                                          int &status, unsigned long long &probes, bool &inserted) {
    inserted = false;
    int idx = tree_find(Q.tab, Q.tmask, Q.nx, Q.ny, Q.nth, e.wx, e.wy, e.wth, probes);
    // Lanes of a group are NOT in lockstep (independent thread scheduling): every lane must have finished
    // reading the tree and its index before the leader modifies them, or a late lane finds the node the
    // leader has just inserted and the group's copies of `n` drift apart.
    g.sync();
    if (idx < 0) {
        if (n >= K) { status = TRRT_ERR_CAPACITY; code = TRRT_IT_NOT_RUN; return -1; }
        idx = n++;
        TRRT_CHECK(idx >= 1 && idx < K);
        inserted = true;
        if (g.gl == 0) {
            Q.nx[idx] = e.wx; Q.ny[idx] = e.wy; Q.nth[idx] = e.wth;
            Q.parent[idx] = -1;
            if (Q.uo) for (int j = 0; j < 5; j++) Q.uo[5 * idx + j] = NAN;
            tree_insert(Q.tab, Q.tmask, e.wx, e.wy, e.wth, idx);
        }
        code = TRRT_IT_NEW_NODE;
    } else code = TRRT_IT_EXISTING_NODE;
    if (idx != near && g.gl == 0) { // rrt.py:187-188
        Q.parent[idx] = near;
        if (Q.uo) {
            Q.uo[5 * idx] = e.usteer; Q.uo[5 * idx + 1] = (e.flags & 1) ? NAN : e.iccx; Q.uo[5 * idx + 2] = (e.flags & 1) ? NAN : e.iccy;
            Q.uo[5 * idx + 3] = (e.flags & 1) ? NAN : e.rad; Q.uo[5 * idx + 4] = e.udist;
        }
    }
    g.sync(); // tree + index writes visible to the whole group
    return idx;
}

// n elements, G lanes, eight independent loads in flight per lane (the copy sits on the critical path of its CTA: the
// other warps wait for this one at the next barrier)
template <int G, typename T>
__device__ __forceinline__ void group_copy(const Group<G> &g, T *__restrict__ dst, const T *__restrict__ src, int n) {
    int i = g.gl;
    for (; i + 7 * G < n; i += 8 * G) {
        T v[8];
#pragma unroll
        for (int k = 0; k < 8; k++) v[k] = src[i + k * G];
#pragma unroll
        for (int k = 0; k < 8; k++) dst[i + k * G] = v[k];
    }
    for (; i < n; i += G) dst[i] = src[i];
}

struct RrtCounters {
    unsigned long long scan, los, lospx, arcpx, arcang, steer, drive, probe;
    unsigned long long ties; // nearest decisions that the reference's sqrt could have taken differently (SURVEY H3), see nearest_tie_audit
};

// The kernels take the argmin of d2 = rn(rn(dx*dx) + rn(dy*dy)); the reference takes np.argmin over sqrt(pow, pow)
// (search.py:15, rrt.py:157), first minimum.  sqrt is monotone, so the two can only differ when a node with a LOWER index
// than the winner has a slightly larger d2 that collapses to the SAME correctly rounded sqrt (then the reference keeps the
// lower index).  Audit (counters mode only): is there a node i < winner with d2_i > best and sqrt(d2_i) == sqrt(best)?
// (Nodes a few ulp apart do occur -- the same point reached along two different arcs -- but their d2 differ by >= 2 ulp
// and the square roots stay distinct.)  G lanes share the loop.  Expected: never -- the tests assert the counter is 0.
template <int G>
__device__ __forceinline__ bool nearest_tie_audit(const Group<G> &g, const double *__restrict__ nx, const double *__restrict__ ny, int winner,
                                                  double best, double qx, double qy, bool shared_query) {
    const double hi = best * (1.0 + 8.881784197001252e-16), sbest = sqrt(best); // 4-ulp window first, the sqrt only inside it
    bool amb = false;
    if (shared_query) { // the group works on ONE query: lanes stride the nodes
        for (int i = g.gl; i < winner; i += G) {
            const double dx = qx - nx[i], dy = qy - ny[i];
            const double d = dx * dx + dy * dy;
            if (d > best && d <= hi && sqrt(d) == sbest) amb = true;
        }
        return g.any(amb);
    }
    for (int i = 0; i < winner; i++) { // one query per lane (speculative window): every lane walks its own prefix
        const double dx = qx - nx[i], dy = qy - ny[i];
        const double d = dx * dx + dy * dy;
        if (d > best && d <= hi && sqrt(d) == sbest) amb = true;
    }
    return amb;
}

// c: the group's counter sums, written to the query's row when a.counters is set; nullptr when the kernel has already summed
// into that row (rrt_kernel_spec)
template <int G>
__device__ __forceinline__ void rrt_finish(const RrtDev &a, int64_t q, const Group<G> &g, const RrtQuery &Q, int K, int iters, int n, int sol,
                                           int status, int nlos, const RrtCounters *c) {
    if (status == TRRT_OK_NOT_FOUND && iters < K - 1) status = TRRT_PAUSED; // the query's stop cut the loop
    if (g.gl == 0) {
        if (Q.it_near || Q.it_new || Q.it_code) {
#pragma unroll 1
            for (int i = iters; i < K - 1; i++) {
                if (Q.it_near) Q.it_near[i] = -1;
                if (Q.it_new) Q.it_new[i] = -1;
                if (Q.it_code) Q.it_code[i] = TRRT_IT_NOT_RUN;
            }
        }
        a.n_nodes[q] = n;
        a.sol[q] = sol;
        a.status[q] = status;
        a.iters[q] = iters;
        if (a.race_group && status == TRRT_OK_FOUND) { // publish to the race group (launcher: q < 2^32)
            const int gi = race_group_of(a, q);
            if (gi >= 0) atomicMin(a.race_key + gi, ((unsigned long long)iters << 32) | (unsigned long long)q);
        }
        if (a.n_los) a.n_los[q] = nlos;
        if (a.counters && c) {
            unsigned long long *o = a.counters + q * 9;
            const unsigned long long v[9] = {c->scan, c->los, c->lospx, c->arcpx, c->arcang, c->steer, c->drive, c->probe, c->ties};
            for (int j = 0; j < 9; j++) o[j] = (a.resume ? o[j] : 0ull) + v[j]; // a resumed query adds to its row
        }
    }
    if (a.row_start) { // packed copy of the rows that exist: one row reservation per query, coalesced copies by the group
        unsigned long long r0 = 0;
        if (g.gl == 0) r0 = atomicAdd(a.pack_rows, (unsigned long long)n);
        r0 = g.bcast(r0, 0);
        group_copy<G>(g, a.px + r0, Q.nx, n); group_copy<G>(g, a.py + r0, Q.ny, n); group_copy<G>(g, a.pth + r0, Q.nth, n);
        group_copy<G>(g, a.pparent + r0, Q.parent, n);
        if (a.pu && Q.uo) group_copy<G>(g, a.pu + 5 * r0, Q.uo, 5 * n);
        if (g.gl == 0) a.row_start[q] = (long long)r0;
    }
}

// Applies the outcome `e` of iteration `it` (nearest node `near`) to the tree; uniform across the group.
// Returns false when the loop must stop (goal reached or the reference would raise).
template <int G>
__device__ __forceinline__ bool rrt_commit(const Group<G> &g, const RrtQuery &Q, const Expand &e, int near, int K, int &n, int &nlos, int &sol,
                                           int &status, int &code, int &newi, RrtCounters &c, bool &inserted) {
    inserted = false;
    c.steer++;
    if (e.code == TRRT_IT_STEER_CONSTRAINT) { code = TRRT_IT_STEER_CONSTRAINT; return true; }
    const int nl = (e.flags >> 4) & 3;
    if (Q.los_log && g.gl == 0) {
        if (nl >= 1) Q.los_log[nlos] = (e.flags >> 6) & 1;
        if (nl >= 2) Q.los_log[nlos + 1] = (e.flags >> 7) & 1;
    }
    nlos += nl;
    c.los += nl; c.lospx += e.lospx; c.arcpx += e.arcpx; c.arcang += e.arcang; c.drive += e.drive;
    if (e.flags & 2) { status = TRRT_ERR_REF_RAISES_DRIVE_NONE; code = TRRT_IT_NOT_RUN; return false; }
    if (e.code == TRRT_IT_ARC_BLOCKED) { code = TRRT_IT_ARC_BLOCKED; return true; }
    newi = rrt_insert<G>(g, Q, e, near, K, n, code, status, c.probe, inserted);
    if (newi < 0) return false;
    if (e.flags & 4) { sol = newi; status = TRRT_OK_FOUND; return false; }
    return true;
}

// ---------------------------------------------------------------------------
// schedule 1: cooperative, one iteration at a time
// ---------------------------------------------------------------------------
template <int G>
__global__ void __launch_bounds__(128) rrt_kernel_coop(const RrtDev a) {
    const Group<G> g;
    const int64_t q = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / G;
    if (q >= a.nq) return; // whole groups leave together
    if (a.resume && !query_resumes<G>(a, q, g)) return; // not written at all
    const int K = a.K;
    RrtQuery Q;
    RrtCounters c = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    int n = 1, nlos = 0, sol = -1, status = TRRT_OK_NOT_FOUND, it0 = 0;
    if (a.resume) rrt_setup_resume<G>(a, q, g, Q, n, it0, nlos);
    else rrt_setup<G>(a, q, g, Q);
    int k;
    for (k = it0 + 1; k <= Q.limit; k++) {
        const int it = k - 1;
        if (a.race_group && it >= race_limit_group<G>(a, q, g, Q.limit)) break; // a member of the race group found the goal by it
        int sx, sy;
        sample_xy(a, Q, it, sx, sy);
        const double qx = (double)sx, qy = (double)sy;
        const double qth = standardangle(__ldg(Q.sth + it));
        int code, near = -1, newi = -1;
        bool go = true;
        if (!Q.m.freespace(sx, sy)) code = TRRT_IT_QRAND_BLOCKED;                                            // rrt.py:148
        else if (tree_find(Q.tab, Q.tmask, Q.nx, Q.ny, Q.nth, qx, qy, qth, c.probe) >= 0) code = TRRT_IT_QRAND_IN_TREE; // rrt.py:151
        else {
            near = nearest_coop<G>(g, Q.nx, Q.ny, n, qx, qy);
            c.scan += (unsigned long long)n;
            if (a.counters) {
                const double bx_ = qx - Q.nx[near], by_ = qy - Q.ny[near];
                if (nearest_tie_audit<G>(g, Q.nx, Q.ny, near, bx_ * bx_ + by_ * by_, qx, qy, true)) c.ties++;
            }
            Expand e;
            expand_from<G>(g, Q.m, a.P, Q.nx[near], Q.ny[near], Q.nth[near], qx, qy, qth, Q.gx, Q.gy, Q.gth, e);
            bool ins;
            go = rrt_commit<G>(g, Q, e, near, K, n, nlos, sol, status, code, newi, c, ins);
        }
        if (g.gl == 0) {
            if (Q.it_near) Q.it_near[it] = near;
            if (Q.it_new) Q.it_new[it] = newi;
            if (Q.it_code) Q.it_code[it] = (uint8_t)code;
        }
        if (!go) {
            if (status == TRRT_OK_FOUND) k++;
            break;
        }
    }
    rrt_finish<G>(a, q, g, Q, K, k - 1, n, sol, status, nlos, &c);
}

// ---------------------------------------------------------------------------
// schedule 0: speculative window of up to G iterations (see the header comment)
//
// Phase A (lane j = iteration k0+j, all lanes in parallel, everything in registers):
//   sample -> freespace(qrand) -> `qrand in G` probe of the snapshot index -> nearest scan over the snapshot ->
//   steer / clearance rays / re-drive / edge raster (expand_from<1>) -> `qnew in G` probe.
// Pass (registers and shuffles only): the lanes that insert a node are walked in iteration order; each one's node is
//   folded into the later lanes (distance-to-nodes-of-this-window minimum, `qrand in G`, `qnew in G`).  New nodes have
//   higher indices than the snapshot, so the snapshot winner keeps ties (first-minimum semantics of np.argmin).  The
//   walk stops at the first lane f whose nearest node is no longer its snapshot winner: what lanes 0..f-1 computed
//   is exactly what the sequential loop computes for them.
// Commit: lanes [0, f) write their results TOGETHER -- node indices by prefix popcount, tree rows, index slots
//   (atomicCAS), parents, logs.  The next window starts at iteration k0 + f with a fresh snapshot, i.e. an iteration
//   whose nearest node was inserted in its own window is simply expanded again one window later, in a full-width pass,
//   instead of being re-expanded by a single lane while the rest of the warp (and, through the lockstep barrier, of the
//   CTA) waits.  Lane 0 has no predecessor in its window, so every window commits at least one iteration.
// ---------------------------------------------------------------------------
constexpr int SCAN_AHEAD = 1024; // prefetch distance of nearest_private, in bytes of each coordinate array
// private fp64 nearest scan over nodes [0, n): every lane of the warp reads the same node (broadcast loads)
__device__ __forceinline__ void nearest_private(const double *__restrict__ nx, const double *__restrict__ ny, int n, double qx, double qy,
                                                double &bd_out, int &bi_out) {
    double bd = INFINITY;
    int bi = 0x7fffffff;
    int i = 0;
#define TRRT_NODE(xv, yv, idx) { double dx = qx - (xv), dy = qy - (yv); double d = dx * dx + dy * dy; if (d < bd) { bd = d; bi = (idx); } }
    if ((((uintptr_t)nx ^ (uintptr_t)ny) & 15) == 0) { // rows equally aligned: 16-byte loads, two nodes each
        if (((uintptr_t)nx & 15) != 0 && n > 0) { TRRT_NODE(nx[0], ny[0], 0); i = 1; }
        const double2 *x2 = reinterpret_cast<const double2 *>(nx + i);
        const double2 *y2 = reinterpret_cast<const double2 *>(ny + i);
        const int pairs = (n - i) >> 1;
        int p = 0;
        for (; p + 1 < pairs; p += 2) {
            // the tree streams from L2 / HBM: ask for the lines SCAN_AHEAD bytes ahead (one request per 128-byte line)
            if ((p & 7) == 0 && p + SCAN_AHEAD / 16 < pairs) { // never beyond the nodes that exist
                asm volatile("prefetch.global.L1 [%0];" ::"l"(x2 + p + SCAN_AHEAD / 16));
                asm volatile("prefetch.global.L1 [%0];" ::"l"(y2 + p + SCAN_AHEAD / 16));
            }
            const double2 xa = x2[p], ya = y2[p], xb = x2[p + 1], yb = y2[p + 1];
            const int b = i + 2 * p;
            TRRT_NODE(xa.x, ya.x, b); TRRT_NODE(xa.y, ya.y, b + 1); TRRT_NODE(xb.x, yb.x, b + 2); TRRT_NODE(xb.y, yb.y, b + 3);
        }
        if (p < pairs) {
            const double2 xa = x2[p], ya = y2[p];
            const int b = i + 2 * p;
            TRRT_NODE(xa.x, ya.x, b); TRRT_NODE(xa.y, ya.y, b + 1);
        }
        i += 2 * pairs;
    }
#pragma unroll 1
    for (; i < n; i++) TRRT_NODE(nx[i], ny[i], i);
#undef TRRT_NODE
    bd_out = bd; bi_out = bi;
}

// The same scan for a full warp on one query, staged through shared memory.  In nearest_private every node costs
// the warp two broadcast loads that each fetch 16 useful bytes and stall on L1/L2 (ncu: 45% of the kernel's
// long-scoreboard stalls sit on those loads, and the CTA barrier then waits for the slowest scan).  Here the warp
// copies the tree tile by tile with cp.async (LDGSTS, 512 coalesced bytes per instruction), two tiles in flight, and
// all lanes read the tile from shared memory (conflict-free broadcast) while the next one is landing.
// TILE_PAIRS: double2 pairs of x (and of y) per tile = 64 nodes (one copy instruction per lane and array); 2 tiles x 2
// arrays x 512 B per warp.  Multiple of 32.  Measured (cfg 3): 32 -> 63.7 ms, 64 -> 65.6 ms (less shared memory, more L1).
constexpr int TILE_PAIRS = 32;
__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gmem_src) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gmem_src) : "memory");
}
#ifdef TRRT_PHASE_PROF
// experiment builds only (profiles/tools/phase_prof.py): per-warp clock64 sums of the phases of a window
__device__ unsigned long long g_phase_prof[24];
#define TRRT_PROF(...) __VA_ARGS__
#else
#define TRRT_PROF(...)
#endif

// Packed-fp32 prefilter of the staged scan.  The fp64 scan costs 6 fp64-pipe and ~11 warp instructions per (sample, node)
// pair.  Here each staged tile is converted once to fp32 coordinates relative to an integer origin, every lane streams it
// against its own sample with f32x2 instructions (FADD2 x2, FMUL2, FFMA2, FMNMX3: ~2.5 instructions per pair, none on the
// fp64 pipe) and keeps one fp32 minimum per block of SCAN_BLOCK nodes.  fp32 only filters: the blocks that can hold the fp64
// winner are rescanned with the fp64 arithmetic of TRRT_NODE, so the result is the same bit for bit.  Those blocks are folded
// in by (d2, index), lexicographically, so the order in which they are rescanned does not matter: the lowest index wins ties.
//
// Error bound, per pair (u = 2^-24, v = 2^-53).  X = x - ox exactly; fx = rn32(rn64(X)), so |fx - X| <= e1 = (u + 1.0001 v) M
// with M the tile's largest |fx| or |fy|.  The sample s = qx - ox is an integer, exact in fp32 (|s| <= 2^24, checked), and
// a = qx - x = s - X exactly.  dxf = rn32(s - fx) satisfies |dxf - a| <= e1 + u' |dxf| (u' = u / (1 - u)), hence
// |dxf^2 - a^2| <= e1^2 + 2 (1 + u') e1 |dxf| + (2u' + u'^2) dxf^2, likewise for y.  With G = dxf^2 + dyf^2, |dxf| + |dyf| <=
// sqrt(2G) and 2 e1 (1 + u') sqrt(2G) <= t G + 2 e1^2 (1 + u')^2 / t for any t > 0:
//     |G - S| <= t G + 2.0001 u G + 2 e1^2 ((1 + u')^2 / t + 1)        (S = a^2 + b^2)
// The scan computes F = rn32(fma(dyf, dyf, rn32(dxf^2))); fused or not, |F - G| <= 2.0001 u G.  The kernel's fp64
// D = rn(rn(dx^2) + rn(dy^2)) with dx = rn(qx - x) satisfies |D - S| <= 4.001 v S.  With t = 2^-16 and G <= F / (1 - 2.0001 u):
//     |F - D| <= SCAN_REL * F + SCAN_ABS * M^2,   SCAN_REL = 2^-15 (needs 1.55e-5), SCAN_ABS = 2^-30 (needs 2^-31 (1 + 2^-15)).
// So over a block whose fp32 minimum is m, every D is >= m (1 - SCAN_REL) - c, and the node attaining m has D <= m (1 +
// SCAN_REL) + c (c = SCAN_ABS * M^2): lower and upper bounds, computed with directed rounding so that they stay bounds.
// tests/test_scan_prefilter.py checks this inequality on emulated pairs (random and adversarial).
//
// Tiles whose |fx| or |fy| exceeds SCAN_FP32_MAX, or is not finite, are not filtered: every lane then scans the whole slice in
// fp64, and so does a lane whose sample is not exact in fp32.  Coordinates near the map (|X| up to 2^20 pixels) keep c below
// 2^10 and F finite.
//
// SCAN_BLOCK: nodes per fp32 block minimum (a divisor of 2 * TILE_PAIRS).  SCAN_LIST: candidate blocks a lane keeps until the
// end of its slice; a block admitted while the list holds SCAN_LIST live candidates is rescanned at once instead (near-equal
// nodes in several blocks: 0.014 blocks per lane-slice on cfg 3).  Measured on B200, cfg 3 (parent fp64 scan 34.4 ms): as
// shipped (rescans one pair at a time) 30.6 ms; with four pairs per rescan step 32.1 ms at SCAN_BLOCK 16, 31.0 ms at 8,
// 34.3 ms at 32, 32.2 ms with SCAN_LIST 2 (profiles/r4/NOTES.md).
constexpr int SCAN_BLOCK = 16, SCAN_LIST = 3;
constexpr float SCAN_REL = 0x1p-15f, SCAN_ABS = 0x1p-30f, SCAN_FP32_MAX = 0x1p20f;
static_assert(TILE_PAIRS == 32, "the conversion pass gives lane l pair l of the tile: the pair its own cp.async staged");
static_assert(SCAN_BLOCK % 2 == 0 && (2 * TILE_PAIRS) % SCAN_BLOCK == 0, "blocks of whole pairs that tile a tile");

__device__ __forceinline__ unsigned long long f32x2_pack(float lo, float hi) {
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
// F of the two nodes of a packed pair: rn(fma(dy, dy, rn(dx * dx))), dx = rn(sx - x), dy = rn(sy - y), for both halves
__device__ __forceinline__ void f32x2_d2(unsigned long long sx2, unsigned long long sy2, unsigned long long x2, unsigned long long y2,
                                         float &d0, float &d1) {
    unsigned long long dx, dy, d;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(dx) : "l"(sx2), "l"(x2));
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(dy) : "l"(sy2), "l"(y2));
    asm("mul.rn.f32x2 %0, %1, %1;" : "=l"(d) : "l"(dx));
    asm("fma.rn.f32x2 %0, %1, %1, %2;" : "=l"(d) : "l"(dy), "l"(d));
    asm("mov.b64 {%0, %1}, %2;" : "=f"(d0), "=f"(d1) : "l"(d));
}

struct ScanStats { // counters of the phase-profile build
    int blocks, rechecked, settled, fp64;
    long long cyc_wait, cyc_settle; // clock64 in cp.async waits, in fp64 rescans
};

// Nodes [lo, n) of the tree (lo = 0: the whole tree); lowest index on ties inside the range.  (ox, oy): integer origin of
// the fp32 coordinates.
__device__ __forceinline__ void nearest_staged(double2 *tile /* [2][2][TILE_PAIRS] of this warp */, const double *__restrict__ nx,
                                               const double *__restrict__ ny, int lo, int n, double qx, double qy, double ox, double oy,
                                               double &bd_out, int &bi_out, ScanStats &st) {
    const int lane = threadIdx.x & 31;
    double bd = INFINITY;
    int bi = 0x7fffffff;
    int i = lo;
    // (d2, index) lexicographic: nodes may be folded in any order, the first minimum wins
#define TRRT_NODE(xv, yv, idx) { double dx = qx - (xv), dy = qy - (yv); double d = dx * dx + dy * dy; if (d < bd || (d == bd && (idx) < bi)) { bd = d; bi = (idx); } }
    if ((((uintptr_t)nx ^ (uintptr_t)ny) & 15) == 0) { // rows equally aligned
        if (((uintptr_t)(nx + i) & 15) != 0 && i < n) { TRRT_NODE(nx[i], ny[i], i); i++; }
        const double2 *x2 = reinterpret_cast<const double2 *>(nx + i);
        const double2 *y2 = reinterpret_cast<const double2 *>(ny + i);
        const int pairs = (n - i) >> 1;
        const int tiles = (pairs + TILE_PAIRS - 1) / TILE_PAIRS;
        // the sample relative to the origin, exact in fp32 (else this lane rescans its slice in fp64)
        const double sxd = qx - ox, syd = qy - oy;
        bool all64 = !(fabs(sxd) <= 0x1p24 && fabs(syd) <= 0x1p24);
        bool wide = false; // warp-uniform: a tile that fp32 cannot filter was seen
        const unsigned long long sx2 = f32x2_pack((float)sxd, (float)sxd), sy2 = f32x2_pack((float)syd, (float)syd);
        // fp64 rescan of block b, from global memory (the slice was just streamed through L2; the fp64 x of the tile in shared
        // memory has been overwritten by the fp32 tile).
        auto settle = [&](int b) {
            const int q0 = b * (SCAN_BLOCK / 2), q1 = q0 + SCAN_BLOCK / 2 < pairs ? q0 + SCAN_BLOCK / 2 : pairs;
            TRRT_CHECK(b >= 0 && q0 < pairs && i + 2 * q1 <= n);
#pragma unroll 1
            for (int p = q0; p < q1; p++) {
                const double2 xa = x2[p], ya = y2[p];
                TRRT_NODE(xa.x, ya.x, i + 2 * p); TRRT_NODE(xa.y, ya.y, i + 2 * p + 1);
            }
        };
        // Candidate list.  U: running minimum of the blocks' upper bounds; an entry holds a block and its lower bound cl.  A
        // block is admitted when cl <= U at the time it is scanned; an entry whose cl has risen above U is free again, and a
        // block admitted to a list of live entries only is rescanned at once.  U only falls, and the winner's block has cl <=
        // D(winner) <= final U <= U at any time: it is admitted when scanned, and then never freed.  A block never admitted,
        // or freed, has every D > final U >= D(winner): no ties with the winner either.
        float U = INFINITY, cl[SCAN_LIST];
        int cb[SCAN_LIST];
#pragma unroll
        for (int s = 0; s < SCAN_LIST; s++) { cl[s] = INFINITY; cb[s] = 0; }
        auto issue = [&](int t) { // lanes copy pairs lane, lane + 32 of tile t (only pairs that exist)
            double2 *bx = tile + (t & 1) * 2 * TILE_PAIRS, *by = bx + TILE_PAIRS;
            const int p0 = t * TILE_PAIRS;
#pragma unroll
            for (int k = 0; k < TILE_PAIRS / 32; k++) {
                const int p = p0 + lane + 32 * k;
                if (p < pairs) { cp_async16(bx + lane + 32 * k, x2 + p); cp_async16(by + lane + 32 * k, y2 + p); }
            }
            asm volatile("cp.async.commit_group;" ::: "memory");
        };
        if (tiles > 0) issue(0);
        for (int t = 0; t < tiles; t++) {
            TRRT_PROF(const long long tw_ = clock64();)
            if (t + 1 < tiles) { issue(t + 1); asm volatile("cp.async.wait_group 1;" ::: "memory"); }
            else asm volatile("cp.async.wait_group 0;" ::: "memory");
            TRRT_PROF(st.cyc_wait += clock64() - tw_;)
            // this lane's pair of tile t has landed (its own copy): convert it in place to fp32 (x0, x1, y0, y1)
            double2 *bx = tile + (t & 1) * 2 * TILE_PAIRS;
            const double2 *by = bx + TILE_PAIRS;
            float4 *f4 = reinterpret_cast<float4 *>(bx);
            const int p0 = t * TILE_PAIRS;
            const int cnt = pairs - p0 < TILE_PAIRS ? pairs - p0 : TILE_PAIRS;
            unsigned mbits = 0;
            if (lane < cnt) {
                const double2 xa = bx[lane], ya = by[lane];
                const float4 f = make_float4((float)(xa.x - ox), (float)(xa.y - ox), (float)(ya.x - oy), (float)(ya.y - oy));
                // max of |f| as bit patterns: NaN sorts above +inf above every finite value
                mbits = max(max(__float_as_uint(fabsf(f.x)), __float_as_uint(fabsf(f.y))), max(__float_as_uint(fabsf(f.z)), __float_as_uint(fabsf(f.w))));
                f4[lane] = f;
            } else f4[lane] = make_float4(0x1p30f, 0x1p30f, 0x1p30f, 0x1p30f); // pads the last block: F ~ 2^61, never a candidate
            mbits = __reduce_max_sync(0xffffffffu, mbits);
            __syncwarp(); // the fp32 tile is complete
            if (mbits > __float_as_uint(SCAN_FP32_MAX)) wide = true;
            if (!wide) {
                const float M = __uint_as_float(mbits), c = __fmul_ru(__fmul_ru(M, M), SCAN_ABS);
                const ulonglong2 *fp = reinterpret_cast<const ulonglong2 *>(f4);
                for (int pb = 0; pb < cnt; pb += SCAN_BLOCK / 2) {
                    float m = INFINITY;
#pragma unroll
                    for (int k = 0; k < SCAN_BLOCK / 2; k++) {
                        const ulonglong2 v = fp[pb + k];
                        float d0, d1;
                        f32x2_d2(sx2, sy2, v.x, v.y, d0, d1);
                        m = fminf(m, fminf(d0, d1));
                    }
                    const float lb = __fmaf_rd(m, 1.0f - SCAN_REL, -c), ub = __fmaf_ru(m, 1.0f + SCAN_REL, c);
                    U = fminf(U, ub);
                    TRRT_PROF(st.blocks++;)
                    if (lb <= U) {
                        const int blk = (2 * (p0 + pb)) / SCAN_BLOCK;
                        bool placed = false;
#pragma unroll
                        for (int s = 0; s < SCAN_LIST; s++)
                            if (!placed && !(cl[s] <= U)) { cl[s] = lb; cb[s] = blk; placed = true; }
                        if (!placed && !all64) { TRRT_PROF(const long long ts_ = clock64();) settle(blk); TRRT_PROF(st.settled++; st.cyc_settle += clock64() - ts_;) }
                    }
                }
            }
            __syncwarp(); // tile t may be overwritten by the copy of tile t + 2
        }
        // exact fp64 rescan of the live candidates, or of the whole slice
        TRRT_PROF(const long long ts_ = clock64();)
        if (all64 || wide) {
            TRRT_CHECK(i + 2 * pairs <= n);
#pragma unroll 1
            for (int p = 0; p < pairs; p++) {
                const double2 xa = x2[p], ya = y2[p];
                TRRT_NODE(xa.x, ya.x, i + 2 * p); TRRT_NODE(xa.y, ya.y, i + 2 * p + 1);
            }
            TRRT_PROF(st.fp64++;)
        } else if (tiles > 0) { // (no tile, no block: U is still +inf and the list empty)
#pragma unroll 1
            for (int r = 0; r < SCAN_LIST; r++) {
                int b = -1; // the entry of slot r, if live (one call site of settle)
#pragma unroll
                for (int s = 0; s < SCAN_LIST; s++) if (s == r && cl[s] <= U) b = cb[s];
                if (b >= 0) { settle(b); TRRT_PROF(st.rechecked++;) }
            }
        }
        TRRT_PROF(st.cyc_settle += clock64() - ts_;)
        i += 2 * pairs;
    }
#pragma unroll 1
    for (; i < n; i++) TRRT_NODE(nx[i], ny[i], i);
#undef TRRT_NODE
    bd_out = bd; bi_out = bi;
}

// Counters launches of rrt_kernel_spec: every lane adds its share straight to the query's row, so no counter is carried
// through the window loop.  Nine per-lane sums would hold 18 registers across the expansion, and a per-warp copy (14 x 72 B)
// does not fit the kernel's 48 KB of static shared memory: with sQ the kernel uses 48 968 of 49 152 bytes.  The group zeroes
// the row when it takes the query: the C ABI has always had the kernel write the whole row, so callers other than
// Planner.rrt need not clear d_counters.
__device__ __forceinline__ void count_add(const RrtDev &a, int64_t q, int k, unsigned long long v) {
    if (v) atomicAdd(a.counters + q * 9 + k, v);
}

// CTA shape of rrt_kernel_spec, also read by its launch: 2 CTAs of 14 warps = 28 warps per SM at 72 registers, so the
// 4 096 queries of cfg 3 are resident at once (4 144 warps), no second wave.  Measured on B200 (cfg 3): 448 x 2 39.4 ms,
// 384 x 2 43.9 ms, 512 x 2 (64 registers) 42.4 ms, 768 x 1 43.0 ms; see profiles/r2/NOTES.md.
constexpr int SPEC_THREADS = 448, SPEC_BLOCKS_PER_SM = 2;

// Lockstep: the expansion code (steer, libm, rays, raster: ~40 KB of SASS) is far larger than an SM's instruction
// cache, and with warps spread over it the instruction fetches of a GPC saturate its shared cache (ncu: gcc
// instruction requests at 85% of peak, SM i-cache hit rate 68%, half of all stall samples "no instruction").
// So the warps of a CTA enter the expansion together: one CTA barrier per window, placed after the (tiny-code)
// nearest scan; the first warp through a code line fetches it for the others (SM i-cache hit rate 89%, gcc at 47%).

template <int G>
__global__ void __launch_bounds__(SPEC_THREADS, SPEC_BLOCKS_PER_SM) rrt_kernel_spec(const RrtDev a) {
    const Group<G> g;
    const Group<1> solo;
    const int K = a.K;
    __shared__ __align__(16) double2 scan_tiles[(G == 32) ? (SPEC_THREADS / 32) * 4 * TILE_PAIRS : 1];
    double2 *scan_tile = scan_tiles + ((G == 32) ? (threadIdx.x >> 5) * 4 * TILE_PAIRS : 0);
    // pooled scan (G == 32): what every warp of the CTA needs to scan a slice of any warp's tree for that warp's samples
    constexpr int NW = SPEC_THREADS / 32;
    static_assert(NW <= 32, "one lane per warp of the CTA in the scan partition");
    __shared__ double2 pool_q[(G == 32) ? NW : 1][32];            // sample of lane l of warp w
    __shared__ int pool_n[(G == 32) ? NW : 1];                    // nodes to scan (0: warp w has nothing to scan)
    __shared__ double pool_d[(G == 32) ? 2 * NW : 1][32];         // partial minima: one slot per (warp, tree) overlap
    __shared__ int pool_i[(G == 32) ? 2 * NW : 1][32];
    const unsigned lane_lt = (1u << g.gl) - 1u;
    // The parameter block is handed to non-inlined device functions by reference.  A reference into the kernel's parameter
    // space would be copied to every thread's local stack (192 bytes); one copy per CTA in shared memory serves all of them
    // (1712 -> 1312 bytes of stack).
    __shared__ BikeParams sP;
    // The query's map, row pointers and goal are the same in every lane of a group.  As per-lane copies they held ~35
    // registers for the whole window and pushed the expansion's live set onto the stack; one copy per warp in shared memory
    // is read where it is needed (the pooled scan reads the other warps' tree pointers from it too).  G < 32 puts several
    // groups in a warp; those instantiations keep a copy per lane.
    // Invariant: warp v writes sQ[v] only in rrt_setup, at the top of a loop trip, i.e. after the previous window's
    // __syncthreads_or; other warps read sQ[v].nx / .ny only in the pooled scan, between the window's two CTA barriers,
    // and only when pool_n[v] > 0.  A write to sQ inside a window would race with those reads.
    __shared__ RrtQuery sQ[(G == 32) ? NW : 1];
    RrtQuery Qlane;
    RrtQuery &Q = (G == 32) ? sQ[threadIdx.x >> 5] : Qlane;
    for (int i = threadIdx.x; i < (int)(sizeof(BikeParams) / 4); i += blockDim.x) reinterpret_cast<int *>(&sP)[i] = reinterpret_cast<const int *>(&a.P)[i];
    __syncthreads();
    // persistent groups: queries differ a lot in length (27% of the cfg-3 queries end early), so each group
    // pulls the next query from a counter instead of owning a fixed one.  One loop trip = one window.
    bool have = false, drained = false;
    int64_t q = 0;
    int n = 1, nlos = 0, sol = -1, status = TRRT_OK_NOT_FOUND, iters = 0, k0 = 0;
    TRRT_PROF(unsigned long long pf[24]; for (int i_ = 0; i_ < 24; i_++) pf[i_] = 0; long long t0_, t1_ = 0, t2_, t3_, t4_ = 0, t5_ = 0;)
    for (;;) {
        while (!have && !drained) { // a resume call skips the queries it does not continue
            unsigned long long qq = 0;
            if (g.gl == 0) qq = atomicAdd(a.next_query, 1ull);
            qq = g.bcast(qq, 0);
            if (qq >= (unsigned long long)a.nq) drained = true;
            else {
                q = (int64_t)qq;
                sol = -1; status = TRRT_OK_NOT_FOUND;
                if (a.resume) {
                    if (!query_resumes<G>(a, q, g)) continue;
                    rrt_setup_resume<G>(a, q, g, Q, n, iters, nlos);
                    k0 = iters;
                } else {
                    if (a.counters && g.gl == 0) for (int j = 0; j < 9; j++) a.counters[q * 9 + j] = 0; // summed into by count_add
                    rrt_setup<G>(a, q, g, Q);
                    n = 1; nlos = 0; iters = 0; k0 = 0;
                }
                have = true;
            }
        }
        // ---------------- phase A, part 1: sample, `qrand in G`, nearest scan
        TRRT_PROF(t0_ = clock64();)
        int pre = TRRT_IT_NOT_RUN; // TRRT_IT_QRAND_BLOCKED, TRRT_IT_NOT_RUN (beyond the last iteration / no query) or -1 = live
        bool q_in_tree = false;    // rrt.py:151 against the snapshot (+ nodes of this window, folded in below)
        int near = -1, exist = -1; // nearest node; index of a tree node equal to qnew, or -1
        int islot = 0;             // where the index lookup of qnew ended (see tree_find_slot)
        double bd = INFINITY, qx = 0, qy = 0, qth = 0;
        unsigned long long probes = 0;
        Expand e;
        e.code = TRRT_IT_NOT_RUN; e.flags = 0; e.lospx = e.arcpx = e.arcang = e.drive = 0;
        e.wx = e.wy = e.wth = NAN; // never equal to a node
        // iterations it < lim run: the query's stop, lowered to its race group's best (sQ is not written in a window)
        const int lim = have ? race_limit_group<G>(a, q, g, Q.limit) : 0;
        if (have) {
            const int my_it = k0 + g.gl;
            if (my_it < lim) { // beyond the query's stop: TRRT_IT_NOT_RUN cuts the window there
                int sx, sy;
                sample_xy(a, Q, my_it, sx, sy);
                qx = (double)sx; qy = (double)sy;
                qth = standardangle(__ldg(Q.sth + my_it));
                if (!Q.m.freespace(sx, sy)) pre = TRRT_IT_QRAND_BLOCKED; // rrt.py:148
                else { pre = -1; q_in_tree = tree_find(Q.tab, Q.tmask, Q.nx, Q.ny, Q.nth, qx, qy, qth, probes) >= 0; }
            }
        }
        const bool live = (pre == -1) && !q_in_tree;
        // ---------------- nearest scan.  One warp per query (G == 32): the trees of a CTA's queries differ in size, some
        // warps have no query any more, and the expansion below is entered by the whole CTA together -- so the CTA scans
        // as a pool.  The trees are cut into tiles of 2 * TILE_PAIRS nodes, the tiles of all trees are laid end to end
        // and every warp takes an equal share of that list (a share overlaps one tree or a few); for each overlap the warp
        // scans its slice for the 32 samples of the warp that owns the tree and leaves the partial minima in shared
        // memory; after the barrier the owner folds the partials of its tree in node order (lowest index on ties).
        int part0 = 0, nparts = 0; // this warp's tree: first partial slot, number of partials
        if (G == 32) {
            const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
            const bool scan_me = have && g.any(live);
            pool_q[wid][lane] = make_double2(qx, qy);
            if (lane == 0) pool_n[wid] = scan_me ? n : 0;
            TRRT_PROF(t1_ = clock64();)
            __syncthreads();
            TRRT_PROF(t4_ = clock64();)
            // lane v describes the tree of warp v: tiles, first tile in the list, first / last warp that scans it, first slot
            constexpr int TN = 2 * TILE_PAIRS;
            const int nv = lane < NW ? pool_n[lane] : 0;
            const int tv = (nv + TN - 1) / TN;
            int cv = tv; // inclusive prefix sum of the tile counts
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, cv, o); if (lane >= o) cv += t; }
            const int T = __shfl_sync(0xffffffffu, cv, 31);
            cv -= tv; // first tile of tree v
            // warp k owns tiles [k*T/NW, (k+1)*T/NW): tile c belongs to warp ((c+1)*NW - 1) / T
            int kf = 0, kl = -1;
            if (tv > 0) { kf = ((cv + 1) * NW - 1) / T; kl = ((cv + tv) * NW - 1) / T; }
            const int npv = kl - kf + 1;
            int bv = npv; // exclusive prefix sum: first partial slot of tree v
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, bv, o); if (lane >= o) bv += t; }
            bv -= npv;
            part0 = __shfl_sync(0xffffffffu, bv, wid);
            nparts = __shfl_sync(0xffffffffu, npv, wid);
            if (T > 0) {
                const int a0 = (wid * T) / NW, a1 = ((wid + 1) * T) / NW; // this warp's share of the tile list
                // (a warp whose share is empty, T < NW, still owes its slot: it leaves +inf there)
                unsigned todo = __ballot_sync(0xffffffffu, tv > 0 && kf <= wid && wid <= kl);
                while (todo) {
                    const int v = __ffs(todo) - 1;
                    todo &= todo - 1;
                    const int c0 = __shfl_sync(0xffffffffu, cv, v), tc = __shfl_sync(0xffffffffu, tv, v);
                    const int n_v = __shfl_sync(0xffffffffu, nv, v), k0v = __shfl_sync(0xffffffffu, kf, v), b0 = __shfl_sync(0xffffffffu, bv, v);
                    const int t0 = (a0 > c0 ? a0 : c0) - c0, t1 = (a1 < c0 + tc ? a1 : c0 + tc) - c0;
                    const int lo = t0 * TN, hi = t1 * TN < n_v ? t1 * TN : n_v;
                    const double2 sq = pool_q[v][lane];
                    double pd = INFINITY;
                    int pi = 0x7fffffff;
                    ScanStats st = {0, 0, 0, 0, 0, 0}; // counted in the phase-profile build only
                    if (lo < hi) nearest_staged(scan_tile, sQ[v].nx, sQ[v].ny, lo, hi, sq.x, sq.y,
                                                (double)(a.W / 2), (double)(a.H / 2), pd, pi, st); // origin: the map centre
                    TRRT_PROF(if (lo < hi) { pf[11] += st.rechecked; pf[12] += st.settled; pf[13] += st.fp64; pf[14]++; pf[15] += st.blocks; pf[5] += st.cyc_wait; pf[6] += st.cyc_settle; })
                    const int slot = b0 + (wid - k0v);
                    TRRT_CHECK(slot >= 0 && slot < 2 * NW && lo >= 0 && hi <= n_v && v < NW);
                    pool_d[slot][lane] = pd; pool_i[slot][lane] = pi;
                }
            }
        } else if (have) nearest_private(Q.nx, Q.ny, live ? n : 0, qx, qy, bd, near);
        // ---------------- CTA barrier: the partial minima are complete, the expansion code is entered together; also the exit test
        TRRT_PROF(t5_ = clock64();)
        if (!__syncthreads_or(have ? 1 : 0)) break;
        TRRT_PROF(t2_ = clock64(); { const unsigned long long s_ = t5_ - t4_; pf[0] += s_; pf[1] += s_ * s_ >> 10; pf[2] += t2_ - t5_; pf[18] += t4_ - t1_; pf[19] += t1_ - t0_; pf[20]++; if (have) pf[10]++; })
        if (!have) continue;
        if (G == 32) { // fold the partial minima of this warp's tree, in node order: the first minimum wins
            const int lane = threadIdx.x & 31;
            TRRT_CHECK(part0 >= 0 && part0 + nparts <= 2 * NW);
            for (int j = 0; j < nparts; j++) {
                const double d = pool_d[part0 + j][lane];
                if (d < bd) { bd = d; near = pool_i[part0 + j][lane]; }
            }
        }
        // ---------------- phase A, part 2: everything after the nearest node
        if (live) {
            TRRT_CHECK(near >= 0 && near < n);
            expand_from<1>(solo, Q.m, sP, Q.nx[near], Q.ny[near], Q.nth[near], qx, qy, qth, Q.gx, Q.gy, Q.gth, e);
            if (e.code == EX_ACCEPT) exist = tree_find_slot(Q.tab, Q.tmask, Q.nx, Q.ny, Q.nth, e.wx, e.wy, e.wth, probes, islot);
        }
        if (a.counters) count_add(a, q, 7, probes);
        g.sync();
        TRRT_PROF(t3_ = clock64(); { const unsigned long long s_ = t3_ - t2_; pf[3] += s_; pf[4] += s_ * s_ >> 10; })
        // ---------------- pass: fold the new nodes forward, find the first lane that has to start over
        unsigned done = 0; // lanes whose outcome inserts a node
        int fs;            // first lane that does not commit in this window
        {
            bool moved = false; // a node of this window is strictly nearer than the snapshot winner
            int last = -1;
            for (;;) {
                const bool livel = pre == -1 && !q_in_tree;
                const bool stop = pre == TRRT_IT_NOT_RUN || (livel && moved);
                const bool insl = g.gl > last && livel && !moved && e.code == EX_ACCEPT && exist < 0;
                const unsigned sm = g.ballot(stop), im = g.ballot(insl);
                fs = sm ? __ffs(sm) - 1 : G;
                const int ni = im ? __ffs(im) - 1 : G;
                if (ni >= fs) break;
                const int idx_i = n + __popc(done);
                done |= 1u << ni;
                last = ni;
                const double vx = g.bcast(e.wx, ni), vy = g.bcast(e.wy, ni), vth = g.bcast(e.wth, ni);
                if (g.gl > ni) {
                    const double dx = qx - vx, dy = qy - vy;
                    const double d = dx * dx + dy * dy;
                    if (d < bd) moved = true;
                    if (qx == vx && qy == vy && qth == vth) q_in_tree = true;                       // rrt.py:151
                    if (exist < 0 && e.wx == vx && e.wy == vy && e.wth == vth) exist = idx_i;        // rrt.py:179
                }
            }
        }
        // a lane before fs that ends the query: the reference raises (Q7), or the goal test passes (rrt.py:191-201)
        bool finished = false;
        int end = fs;
        {
            const bool livel = pre == -1 && !q_in_tree;
            const unsigned tm = g.ballot(livel && ((e.flags & 2) || (e.code == EX_ACCEPT && (e.flags & 4)))) & ((fs >= 32) ? 0xffffffffu : ((1u << fs) - 1u));
            if (tm) {
                const int t = __ffs(tm) - 1;
                end = t + 1;
                done &= (end >= 32) ? 0xffffffffu : ((1u << end) - 1u);
                finished = true;
            }
        }
        // ---------------- commit: lanes [0, end) write their results together
        {
            const bool inseg = g.gl < end;
            const bool livel = inseg && pre == -1 && !q_in_tree;
            const int nl = (livel && e.code != TRRT_IT_STEER_CONSTRAINT) ? ((e.flags >> 4) & 3) : 0; // rays of this iteration
            const unsigned m1 = g.ballot(nl >= 1), m2 = g.ballot(nl >= 2);
            int code = TRRT_IT_NOT_RUN, near_j = -1, newi = -1;
            bool edge = false; // this lane records an edge: cameFrom[newi] = (near, u)  (rrt.py:187-188)
            if (inseg) {
                if (pre != -1) code = TRRT_IT_QRAND_BLOCKED;        // rrt.py:148
                else if (q_in_tree) code = TRRT_IT_QRAND_IN_TREE;  // rrt.py:151
                else {
                    near_j = near;
                    const int before = __popc(done & lane_lt); // nodes inserted by the earlier lanes of the window
                    if (a.counters) {
                        count_add(a, q, 0, (unsigned long long)(n + before)); count_add(a, q, 5, 1);
                        if (nearest_tie_audit<1>(solo, Q.nx, Q.ny, near, bd, qx, qy, false)) count_add(a, q, 8, 1); // window nodes have higher indices
                    }
                    if (e.code == TRRT_IT_STEER_CONSTRAINT) code = TRRT_IT_STEER_CONSTRAINT; // rrt.py:166
                    else {
                        if (Q.los_log) {
                            const int pos = nlos + __popc(m1 & lane_lt) + __popc(m2 & lane_lt);
                            TRRT_CHECK(pos >= 0 && pos + nl <= 2 * (K - 1));
                            if (nl >= 1) Q.los_log[pos] = (e.flags >> 6) & 1;
                            if (nl >= 2) Q.los_log[pos + 1] = (e.flags >> 7) & 1;
                        }
                        if (a.counters) {
                            count_add(a, q, 1, nl); count_add(a, q, 2, e.lospx); count_add(a, q, 3, e.arcpx); count_add(a, q, 4, e.arcang);
                            count_add(a, q, 6, e.drive);
                        }
                        if (e.flags & 2) code = TRRT_IT_NOT_RUN;                              // rrt.py:170-171 raises
                        else if (e.code == TRRT_IT_ARC_BLOCKED) code = TRRT_IT_ARC_BLOCKED;   // rrt.py:174
                        else if (exist >= 0) { code = TRRT_IT_EXISTING_NODE; newi = exist; edge = newi != near; } // rrt.py:179 false
                        else { // rrt.py:179-180: a new vertex
                            newi = n + before;
                            TRRT_CHECK(newi >= 1 && newi < K);
                            code = TRRT_IT_NEW_NODE;
                            edge = true; // its nearest node is an older one
                            Q.nx[newi] = e.wx; Q.ny[newi] = e.wy; Q.nth[newi] = e.wth;
                            tree_insert_cas(Q.tab, Q.tmask, islot, newi);
                        }
                    }
                }
                const int it = k0 + g.gl;
                TRRT_CHECK(it >= 0 && it < K - 1);
                if (Q.it_near) Q.it_near[it] = near_j;
                if (Q.it_new) Q.it_new[it] = newi;
                if (Q.it_code) Q.it_code[it] = (uint8_t)code;
            }
            // cameFrom[qnew] is overwritten by every later edge to the same node (rrt.py:188; equal qnew are common: a
            // clamped steer over the maximum distance depends only on the nearest node and the turn direction), so of the
            // lanes of the window that target one node the last one writes
            if (G > 1) {
                const unsigned peers = __match_any_sync(g.mask, edge ? newi : ~(int)(threadIdx.x & 31));
                if (edge && (peers >> (threadIdx.x & 31)) > 1u) edge = false; // a later lane records its edge to the same node
            }
            if (edge) {
                Q.parent[newi] = near;
                if (Q.uo) {
                    const bool st = e.flags & 1;
                    Q.uo[5 * newi] = e.usteer; Q.uo[5 * newi + 1] = st ? NAN : e.iccx; Q.uo[5 * newi + 2] = st ? NAN : e.iccy;
                    Q.uo[5 * newi + 3] = st ? NAN : e.rad; Q.uo[5 * newi + 4] = e.udist;
                }
            }
            nlos += __popc(m1) + __popc(m2);
            n += __popc(done);
            iters = k0 + end;
            if (finished) {
                if (g.bcast(e.flags & 2, end - 1)) { status = TRRT_ERR_REF_RAISES_DRIVE_NONE; iters = k0 + end - 1; } // the iteration that raises is not counted
                else { sol = g.bcast(newi, end - 1); status = TRRT_OK_FOUND; }
            }
            TRRT_PROF({ pf[16]++; pf[17] += end; })
        }
        g.sync(); // tree and index writes of this window are visible to every lane's next phase A
        TRRT_PROF({ const unsigned long long s_ = clock64() - t3_; pf[7] += s_; pf[8] += s_ * s_ >> 10; const unsigned long long w_ = clock64() - t2_; pf[9] += w_ * w_ >> 10; })
        k0 += end;
        if (finished || k0 >= lim) { // query finished or paused
            rrt_finish<G>(a, q, g, Q, K, iters, n, sol, status, nlos, nullptr);
            g.sync();
            have = false;
        }
    }
    // slots 5, 6, 11-15 are per lane (scan prefilter: cycles in cp.async waits and in fp64 rescans; rechecked candidates, blocks
    // rescanned at admission, fp64 slices, slices, blocks), the others per warp
    TRRT_PROF(for (int i_ = 0; i_ < 24; i_++) if (pf[i_] && ((threadIdx.x & 31) == 0 || (i_ == 5 || i_ == 6 || (i_ >= 11 && i_ <= 15)))) atomicAdd(&g_phase_prof[i_], pf[i_]);)
}

} // namespace trrt
