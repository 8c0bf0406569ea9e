/*
 * rrt_continue.c -- TEST INFRASTRUCTURE: the C parity oracle's RRT loop (oracle/trrt_oracle.c, orc_rrt, rrt.py:141-201)
 * continued from a given state, for the tests of tree repair (tests/test_tree_repair.py).
 *
 * The oracle itself stays as it is: this file includes it, so steer, drive, the clearance rays, getArc and the nearest
 * scan are the oracle's own functions, and restates orc_rrt's loop with two extra inputs, the tree it starts from (n0
 * nodes instead of the planted start) and the first iteration it0.  tests/test_tree_repair.py pins the restatement:
 * orc_rrt with K' = j + 1 followed by trc_rrt_continue from j equals one orc_rrt with K, logs included.  The margin audit
 * of orc_rrt is left out.  Built by tests/rrt_continue.py with the oracle's compiler flags.
 */
#include "../oracle/trrt_oracle.c"

/*
 * The tree in node_x/y/th, parent, u (capacity K, 1 <= n0 <= K nodes), no solution, next iteration it0
 * (0 <= it0 <= K-1: samples it0 .. K-2 of sxy / sth are consumed).  Outputs as orc_rrt; the logs are written for
 * iterations >= it0 only, and n_los counts the continuation's lineofsight calls.  Returns the status, -1 for bad input.
 */
int trc_rrt_continue(const uint8_t *grid, int H, int W, const orc_params *P, int K, const double *goal, const int32_t *sxy,
                     const double *sth, double *node_x, double *node_y, double *node_th, int32_t *parent, double *u,
                     int32_t *it_near, int32_t *it_new, uint8_t *it_code, int32_t n0, int32_t it0, int32_t *n_nodes,
                     int32_t *sol, int32_t *iters_run, uint8_t *los_log, int64_t los_cap, int64_t *n_los) {
    if (n0 < 1 || n0 > K || it0 < 0 || it0 > K - 1) return -1;
    orc_map m = {grid, H, W};
    g_aud = NULL;
    double gx = goal[0], gy = goal[1], gth = standardangle(goal[2]);
    int n = n0;
    int64_t nl = 0;
    *sol = -1;
    int status = ORC_OK_NOT_FOUND;
    int k;
    for (k = it0 + 1; k < K; k++) {
        int it = k - 1;
        if (it_near) it_near[it] = -1;
        if (it_new) it_new[it] = -1;
        double qx = (double)sxy[2 * it], qy = (double)sxy[2 * it + 1];
        double qth = standardangle(sth[it]);
        if (!freespace_i(&m, (long)sxy[2 * it], (long)sxy[2 * it + 1])) { if (it_code) it_code[it] = ORC_IT_QRAND_BLOCKED; continue; }
        int dup = 0;
        for (int i = 0; i < n; i++) if (node_x[i] == qx && node_y[i] == qy && node_th[i] == qth) { dup = 1; break; }
        if (dup) { if (it_code) it_code[it] = ORC_IT_QRAND_IN_TREE; continue; }
        int near = (int)orc_nearest(node_x, node_y, n, qx, qy);
        if (it_near) it_near[it] = near;
        double nx = node_x[near], ny = node_y[near], nth = node_th[near];
        steer_out s; steer(P, nx, ny, nth, qx, qy, qth, &s);
        double wx = s.x, wy = s.y, wth = s.theta;
        double us = standardangle(s.steer);
        if (us < P->leftconstraint || us > P->rightconstraint) { if (it_code) it_code[it] = ORC_IT_STEER_CONSTRAINT; continue; }
        /* rrt.py:169 short-circuit `or` chain */
        int ok = valid_d(&m, wx, wy);
        if (ok) {
            ok = clearance_ray(&m, wx, wy, wth, P->bikelength);
            if (los_log && nl < los_cap) los_log[nl] = (uint8_t)ok;
            nl++;
        }
        if (ok) {
            ok = clearance_ray(&m, wx, wy, wth, P->bikelength * P->frontclearance);
            if (los_log && nl < los_cap) los_log[nl] = (uint8_t)ok;
            nl++;
        }
        double udist = s.dist;
        if (!ok) {
            udist = s.dist / 3;
            if (s.straight) { status = ORC_ERR_REF_RAISES_DRIVE_NONE; break; } /* arclength_to_angle(None, ..) TypeError */
            drive(P, nx, ny, nth, s.steer, s.iccx, s.iccy, s.rad, udist, &wx, &wy, &wth);
        }
        pixlist arc = {0};
        get_arc(&m, &arc, nx, ny, wx, wy, s.steer, s.iccx, s.iccy, s.rad, s.straight);
        int blocked = 0;
        for (size_t i = 0; i < arc.n; i++) if (!freespace_i(&m, arc.xy[2 * i], arc.xy[2 * i + 1])) { blocked = 1; break; }
        free(arc.xy);
        if (blocked) { if (it_code) it_code[it] = ORC_IT_ARC_BLOCKED; continue; }
        int idx = -1;
        for (int i = 0; i < n; i++) if (node_x[i] == wx && node_y[i] == wy && node_th[i] == wth) { idx = i; break; }
        if (idx < 0) {
            if (n >= K) { status = ORC_ERR_CAPACITY; break; }
            idx = n++;
            node_x[idx] = wx; node_y[idx] = wy; node_th[idx] = wth; parent[idx] = -1;
            for (int j = 0; j < 5; j++) u[5 * idx + j] = NAN;
            if (it_code) it_code[it] = ORC_IT_NEW_NODE;
        } else if (it_code) it_code[it] = ORC_IT_EXISTING_NODE;
        if (it_new) it_new[it] = idx;
        if (idx != near) { /* qnew != qnear (value equality == index equality, keys are unique) */
            parent[idx] = near;
            u[5 * idx + 0] = s.steer; u[5 * idx + 1] = s.iccx; u[5 * idx + 2] = s.iccy; u[5 * idx + 3] = s.rad; u[5 * idx + 4] = udist;
        }
        double diff = anglediff(wth, gth);
        if (l2norm(wx, wy, gx, gy) < P->tol_xy && fabs(diff) < P->tol_ang) { *sol = idx; status = ORC_OK_FOUND; k++; break; }
    }
    *n_nodes = n;
    *iters_run = k - 1;
    if (it_code) for (int i = k - 1; i < K - 1; i++) { it_code[i] = ORC_IT_NOT_RUN; if (it_near) it_near[i] = -1; if (it_new) it_new[i] = -1; }
    if (n_los) *n_los = nl;
    return status;
}
