// trrt_lane.cuh -- single-lane versions of the ray and arc tests, used where one lane owns one
// RRT iteration (speculative schedule, trrt_rrt.cuh).  Same results as los_group<G> / arc_blocked<G>
// (trrt_device.cuh, trrt_bike.cuh), organised for a lane working alone:
//   * los_lane: literal running-error Bresenham (search.py:58-94), no division;
//   * arc_blocked_lane: 32-bit midpoint-circle rows (DESIGN.md 8.2) restricted to the bounding box of
//     the arc's annular sector, so a long-radius arc costs ~its length in pixel tests instead of the
//     image side (rows outside the box cannot hold a pixel that getArc keeps, DESIGN.md 8.4).
#pragma once
#include "trrt_bike.cuh"

namespace trrt {

// The single-lane ray / raster functions are real calls; they take the grid BY VALUE (four words in registers): by reference the
// caller's copy is forced into local memory (cfg 3: 35.2 -> 34.1 ms).
// search.lineofsight (search.py:35-94) by one lane.  Its pixel count, max(|dx|,|dy|)+1 for in-bounds rays, is los_lane_pixels:
// through a pointer parameter the caller's counter lived on its stack.
__device__ __forceinline__ int los_lane_pixels(const Grid &m, long long ax, long long ay, long long bx, long long by) {
    if (!m.inb(ax, ay) || !m.inb(bx, by)) return 0;
    const long long dx = bx > ax ? bx - ax : ax - bx, dy = by > ay ? by - ay : ay - by;
    return (int)(dx > dy ? dx : dy) + 1;
}
__device__ __noinline__ bool los_lane(const Grid m, long long ax, long long ay, long long bx, long long by) {
    if (!m.inb(ax, ay) || !m.inb(bx, by)) return false;
    int x0 = (int)ax, y0 = (int)ay, x1 = (int)bx, y1 = (int)by;
    const int adx = abs(x1 - x0), ady = abs(y1 - y0);
    const bool low = ady < adx; // search.py:47
    if (low ? (x0 > x1) : (y0 > y1)) { int t = x0; x0 = x1; x1 = t; t = y0; y0 = y1; y1 = t; }
    const int dmaj = low ? adx : ady, dmin = low ? ady : adx;
    const int step = low ? ((y1 < y0) ? -1 : 1) : ((x1 < x0) ? -1 : 1);
    int D = 2 * dmin - dmaj; // search.py:66 / :85
    int aa = low ? x0 : y0, bb = low ? y0 : x0;
    const int aend = aa + dmaj;
    for (; aa <= aend; aa++) {
        const int px = low ? aa : bb, py = low ? bb : aa;
        if (!m.free_nb(px, py)) return false;
        if (D > 0) { bb += step; D -= 2 * dmaj; }
        D += 2 * dmin;
    }
    return true;
}

// largest x >= 0 with x*(x-1) < c, 0 < c < 2^31 (32-bit version of circle_x)
__device__ __forceinline__ int circle_x32(int c) {
    int x = (int)((1.0 + sqrt(1.0 + 4.0 * (double)c)) * 0.5);
    while (x * (x - 1) >= c) --x;
    while ((x + 1) * x < c) ++x;
    return x;
}

#define TRRT_LANE_RMAX 46000 /* r*r must fit 31 bits */

// Outcome of arc_blocked_lane, returned by value (in registers): through pointer parameters the caller's counters lived on
// its stack.
struct ArcLane {
    bool blocked;
    int cand_px, angle_tests; // counters: candidate pixels inside the box, blocked pixels given the angular test
};

// rrt.py:173-174 for a curved edge, one lane: is any pixel of getArc(begin, land, u) not free?
__device__ __noinline__ ArcLane arc_blocked_lane(const Grid m, double bx, double by, double lx, double ly, double usteer, double iccx,
                                                 double iccy, double rad) {
    ArcLane o = {false, 0, 0};
    const long long xc_ = trunc_ll(iccx), yc_ = trunc_ll(iccy), r_ = trunc_ll(rad);
    if (!(r_ < TRRT_LANE_RMAX)) { // enormous radius (cond() allows up to ~1e6): generic 64-bit raster
        const Group<1> solo;
        unsigned long long a = 0, b = 0;
        o.blocked = arc_blocked_impl<1, long long>(solo, m, bx, by, lx, ly, usteer, iccx, iccy, xc_, yc_, r_, &a, &b);
        o.cand_px = (int)a; o.angle_tests = (int)b;
        return o;
    }
    ArcTest A;
    A.iccx = iccx; A.iccy = iccy; A.usteer = usteer;
    A.u1x = bx - iccx; A.u1y = by - iccy;
    A.u2x = lx - iccx; A.u2y = ly - iccy;
    A.n1 = A.u1x * A.u1x + A.u1y * A.u1y;
    A.n2 = A.u2x * A.u2x + A.u2y * A.u2y;
    {
        int sd = (usteer < 0) ? cross_sign(A.u2x, A.u2y, A.u1x, A.u1y, A.n1 * A.n2) : cross_sign(A.u1x, A.u1y, A.u2x, A.u2y, A.n1 * A.n2);
        A.diff_lt_180 = (sd == 0) ? -1 : (sd > 0 ? 1 : 0);
        A.ready = true;
    }
    // ---- bounding box (image coordinates) of every pixel getArc can keep: the raster pixels lie in the annulus
    // rad-3.2 < |p - icc| < rad+2.2 (centre and radius are truncated, the raster is within 0.71 of its circle), and
    // when the span is below 180 degrees they lie in the convex cone spanned by begin-icc and land-icc.
    const double rout = rad + 2.5, rin = fmax(rad - 3.5, 0.0);
    double xlo = -rout, xhi = rout, ylo = -rout, yhi = rout;
    // begin and land both lie on the circle (rad = |begin - icc| by construction, land is begin rotated about icc), so
    // u / rad is their direction; if that ever failed by more than rounding the full box is used
    const double rr2 = rad * rad;
    if (A.diff_lt_180 == 1 && rad > 0.0 && fabs(A.n1 - rr2) <= 1e-6 * rr2 && fabs(A.n2 - rr2) <= 1e-6 * rr2) {
        const double inv = 1.0 / rad, kin = rin * inv, kout = rout * inv;
        // extent of the two boundary rays between the radii: a coordinate c of u spans [c*kin, c*kout] (or reversed)
        const double x1a = A.u1x * (A.u1x < 0 ? kout : kin), x1b = A.u1x * (A.u1x < 0 ? kin : kout);
        const double x2a = A.u2x * (A.u2x < 0 ? kout : kin), x2b = A.u2x * (A.u2x < 0 ? kin : kout);
        const double y1a = A.u1y * (A.u1y < 0 ? kout : kin), y1b = A.u1y * (A.u1y < 0 ? kin : kout);
        const double y2a = A.u2y * (A.u2y < 0 ? kout : kin), y2b = A.u2y * (A.u2y < 0 ? kin : kout);
        xlo = x1a < x2a ? x1a : x2a; xhi = x1b > x2b ? x1b : x2b;
        ylo = y1a < y2a ? y1a : y2a; yhi = y1b > y2b ? y1b : y2b;
        // axis directions inside the cone reach the outer radius (sign convention of arc_keeps_pixel)
        const double sg = (usteer > 0) ? 1.0 : -1.0;
        const double ax_ = sg * A.u1x, ay_ = sg * A.u1y, bx_ = sg * A.u2x, by_ = sg * A.u2y;
        if (ay_ <= 0 && by_ >= 0) xhi = rout;
        if (ay_ >= 0 && by_ <= 0) xlo = -rout;
        if (ax_ >= 0 && bx_ <= 0) yhi = rout;
        if (ax_ <= 0 && bx_ >= 0) ylo = -rout;
        const double pad = 0.5; // directions are rounded; half a pixel dwarfs that
        xlo -= pad; xhi += pad; ylo -= pad; yhi += pad;
    }
    // clip to the image: valid() is x < shape[0], y < shape[1] (square maps)
    const double fxlo = fmax(0.0, floor(iccx + xlo)), fxhi = fmin((double)(m.H - 1), ceil(iccx + xhi));
    const double fylo = fmax(0.0, floor(iccy + ylo)), fyhi = fmin((double)(m.W - 1), ceil(iccy + yhi));
    if (!(fxlo <= fxhi) || !(fylo <= fyhi)) return o; // nothing of the arc can be inside the image
    const int xc = (int)xc_, yc = (int)yc_, r = (int)r_; // box non-empty => the centre is within rout of the image
    const int oxlo = (int)fxlo - xc, oxhi = (int)fxhi - xc, oylo = (int)fylo - yc, oyhi = (int)fyhi - yc;
    const int tmax = (int)circle_tmax(r_);
    const int rr = r * r;
#pragma unroll 1
    for (int k = 0; k < 4; k++) {
        // kind 0: (xc +- x_t, yc + t)   kind 1: (xc +- x_t, yc - t)   kind 2: (xc + t, yc +- x_t)   kind 3: (xc - t, yc +- x_t)
        int tlo, thi, mlo, mhi;
        if (k == 0) { tlo = oylo; thi = oyhi; mlo = oxlo; mhi = oxhi; }
        else if (k == 1) { tlo = -oyhi; thi = -oylo; mlo = oxlo; mhi = oxhi; }
        else if (k == 2) { tlo = oxlo; thi = oxhi; mlo = oylo; mhi = oyhi; }
        else { tlo = -oxhi; thi = -oxlo; mlo = oylo; mhi = oyhi; }
        const int ta = tlo < 0 ? 0 : tlo, tb = thi > tmax ? tmax : thi;
        if (tb < ta) continue;
        // x_t lies in (t, r]: can +x_t or -x_t fall into [mlo, mhi] at all?
        const bool plus_ok = (mhi > ta) && (mlo <= r), minus_ok = (-mlo > ta) && (-mhi <= r);
        if (!plus_ok && !minus_ok) continue;
        o.cand_px += (tb - ta + 1) * ((plus_ok ? 1 : 0) + (minus_ok ? 1 : 0));
        int xt = (ta == 0) ? r : circle_x32(rr - ta * ta); // x_0 = r
        for (int t = ta; t <= tb; t++) {
            const int c = rr - t * t;
            while (xt * (xt - 1) >= c) --xt;
#pragma unroll
            for (int s = 0; s < 2; s++) {
                if (!(s ? minus_ok : plus_ok)) continue;
                const int sx = s ? -xt : xt;
                if (sx < mlo || sx > mhi) continue;
                const int px = (k < 2) ? xc + sx : (k == 2 ? xc + t : xc - t);
                const int py = (k < 2) ? (k == 0 ? yc + t : yc - t) : yc + sx;
                if (!m.free_nb(px, py)) { // inside the image by construction of the box
                    o.angle_tests++;
                    if (arc_keeps_pixel(A, bx, by, lx, ly, (long long)px, (long long)py)) { o.blocked = true; return o; }
                }
            }
        }
    }
    // diagonal-gap pixels (search.py:124-138): only a blocked one inside the box can matter, and only then is the
    // `drawmore` condition (no 4-neighbour of (xc+rnd, yc+rnd) is an emitted raster pixel) evaluated
    const long long rnd = py_round((double)r_ * 0.5 * sqrt(2.0));
    int drawmore = -1;
#pragma unroll 1
    for (int i = 0; i < 4; i++) { // (+,+) (-,-) (+,-) (-,+)
        const long long ox = (i == 0 || i == 2) ? rnd : -rnd, oy = (i == 0 || i == 3) ? rnd : -rnd;
        if (ox < oxlo || ox > oxhi || oy < oylo || oy > oyhi) continue;
        const int px = xc + (int)ox, py = yc + (int)oy;
        if (m.free_nb(px, py)) continue;
        if (drawmore < 0) {
            drawmore = 1;
            const int nx[4] = {1, -1, 0, 0}, ny[4] = {0, 0, 1, -1};
#pragma unroll
            for (int j = 0; j < 4; j++) {
                long long a = rnd + nx[j], b = rnd + ny[j];
                if (m.inb(xc_ + a, yc_ + b) && circle_member(r_, a, b)) drawmore = 0;
            }
        }
        if (!drawmore) break;
        o.angle_tests++;
        if (arc_keeps_pixel(A, bx, by, lx, ly, (long long)px, (long long)py)) { o.blocked = true; return o; }
    }
    return o;
}

} // namespace trrt
