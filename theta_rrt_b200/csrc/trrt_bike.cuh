// trrt_bike.cuh -- scalar fp64 device functions of the kinematic-bicycle RRT:
// angle helpers (rrt.py:9-14,42-51,70-77,108-115), steer (rrt.py:306-541),
// drive (rrt.py:272-304), clearance rays (rrt.py:208-222) and the arc
// collision raster (search.py:96-182).
//
// Operation order follows the reference statement by statement; where the
// reference's compiled dependencies contract a multiply-add (scipy
// Rotation.apply, np.dot, np.linalg.norm, LAPACK dgesv) an explicit fma() is
// used, everything else is compiled with -fmad=false.  sin/cos/atan2 come from
// trrt_libm.h so results are bit-identical to the host oracle.
#pragma once
#include "trrt_device.cuh"

namespace trrt {

#define TRRT_PI 3.141592653589793 /* np.pi */

// Rotation about z by a fixed angle: the matrix scipy's Rotation.apply builds (m11 == m00).
struct Rot {
    double m00, m01, m10;
};

struct BikeParams {
    int thetastar, forwardonly;
    double bikelength, leftconstraint, rightconstraint, frontclearance, maxdrivedist, tol_xy, tol_ang, weightxy;
    // from_euler('z', a) for the angles the reference uses as literals or parameters (rrt.py:333, :412, :280,
    // :379, :383): built once on the host by rot_make(), i.e. by the very code the device would run, so the
    // kernels save five sin/cos evaluations per steer without changing a bit of the result
    Rot r90, rm90, r180, rleft, rright;
};

// rrt.py:9-14
__device__ __forceinline__ double standardangle(double a) {
    while (a > 180) a = a - 360;
    while (a <= -180) a = a + 360;
    return a;
}

// scipy Rotation.from_euler('z', deg, degrees=True) -> quaternion (0,0,z,w)
__device__ __forceinline__ void quat_z(double deg, double &z, double &w) {
    double h = (deg * (TRRT_PI / 180.0)) / 2.0;
    const tl_sc r = tl_sincos_v(h);
    z = r.s; w = r.c;
}

// Rotation.from_euler('z',deg,degrees=True).as_matrix(), the entries apply() needs
__host__ __device__ __forceinline__ Rot rot_from_quat(double z, double w) {
    double z2 = z * z, w2 = w * w, zw = z * w;
    Rot R;
    R.m00 = -z2 + w2;
    R.m01 = 2 * (0.0 - zw);
    R.m10 = 2 * (0.0 + zw);
    return R;
}
__host__ __device__ __forceinline__ Rot rot_make(double deg) {
    double h = (deg * (TRRT_PI / 180.0)) / 2.0;
    const tl_sc r = tl_sincos_v(h);
    return rot_from_quat(r.s, r.c);
}
// Rotation.apply([vx,vy,0])[:2] (the compiled backend contracts the dot products)
__device__ __forceinline__ void rot_apply(const Rot &R, double vx, double vy, double &ox, double &oy) {
    ox = fma(R.m00, vx, R.m01 * vy);
    oy = fma(R.m10, vx, R.m00 * vy);
}
// Rotation.from_euler('z',deg,degrees=True).apply([vx,vy,0])[:2].  Inlined (one tl_sincos_v call and six flops): as a call
// its two results came back through the caller's stack (cfg-3 kernel, mean of 5: 28.94 ms inlined, 29.48 ms as a call).
__device__ __forceinline__ void rotz(double deg, double vx, double vy, double &ox, double &oy) {
    Rot R = rot_make(deg);
    rot_apply(R, vx, vy, ox, oy);
}

// rrt.py:73-77 (np.dot contracts: fma(v1y, v2y, v1x*v2x))
__device__ __noinline__ double anglebetween(double v1x, double v1y, double v2x, double v2y) {
    double dot = fma(v1y, v2y, v1x * v2x);
    double det = v2x * v1y - v1x * v2y;
    return standardangle(tl_atan2(det, dot) * (180.0 / TRRT_PI));
}

// rrt.py:108-115 given the two quaternions (so callers can reuse them)
__device__ __noinline__ double anglediff_q(double s1, double c1, double s2, double c2) {
    double ns1 = -s1;
    double qz = c1 * s2 + c2 * ns1;
    double qw = c1 * c2 - ns1 * s2;
    double n = sqrt(qz * qz + qw * qw);
    qz = qz / n;
    qw = qw / n;
    double hs = tl_atan2(qz, qw);
    double ang = hs + hs;
    if (ang < -TRRT_PI) ang += 2 * TRRT_PI;
    else if (ang > TRRT_PI) ang -= 2 * TRRT_PI;
    return ang * (180.0 / TRRT_PI);
}
__device__ __forceinline__ double anglediff(double a1, double a2) {
    double s1, c1, s2, c2;
    quat_z(a1, s1, c1);
    quat_z(a2, s2, c2);
    return anglediff_q(s1, c1, s2, c2);
}

__device__ __noinline__ double norm2(double x, double y) { return sqrt(fma(y, y, x * x)); } // np.linalg.norm

// rrt.py:42-46
__device__ __forceinline__ void linefrompoints(double px, double py, double qx, double qy, double &a, double &b, double &c) {
    a = qy - py;
    b = px - qx;
    c = a * px + b * py;
}
// rrt.py:48-51 (angle >= 0 at the only call site, rrt.py:482)
__device__ __forceinline__ double angle_to_arclength(double radius, double angle) {
    while (angle < 0) angle = angle + 360;
    return (TRRT_PI * 2 * radius) * angle / 360;
}
// rrt.py:70-71
__device__ __forceinline__ double arclength_to_angle(double radius, double arclength) {
    return arclength * 360 / (TRRT_PI * 2 * radius);
}

// np.linalg.solve, 2x2 (dgesv: partial pivoting, reciprocal-pivot scaling). false = LinAlgError.  Inlined at its two call
// sites in steer(): as a call its results came back through the caller's stack (cfg 3: 28.94 ms inlined, 29.70 ms as a call).
__device__ __forceinline__ bool solve2(double a1, double b1, double a2, double b2, double c1, double c2, double &x1, double &x2) {
    if (fabs(a2) > fabs(a1)) {
        double t;
        t = a1; a1 = a2; a2 = t;
        t = b1; b1 = b2; b2 = t;
        t = c1; c1 = c2; c2 = t;
    }
    if (a1 == 0.0) return false;
    double l = a2 * (1.0 / a1);
    double u22 = fma(-l, b1, b2);
    if (u22 == 0.0) return false;
    double y2 = fma(-l, c1, c2);
    x2 = y2 / u22;
    x1 = fma(-b1, x2, c1) / a1;
    return true;
}
// np.linalg.cond (2-norm) of [[a,b],[c,d]]
__device__ __noinline__ double cond2(double a, double b, double c, double d) {
    double E = a * a + b * b + c * c + d * d;
    double D = fabs(a * d - b * c);
    double disc = E * E - 4 * D * D;
    if (disc < 0) disc = 0;
    double smax2 = (E + sqrt(disc)) / 2;
    if (D == 0.0) return INFINITY;
    return smax2 / D;
}

struct Steer {
    double x, y, theta;                  // landing state
    double steer, iccx, iccy, rad, dist; // u
    double bfx, bfy;                     // Rz(theta)*[bikelength,0] of the origin bike (rrt.py:328-330), reused by drive()
    bool straight;                       // u = (0, None, None, 1)
};

// rrt.py:526-541.  Inlined at its two call sites in steer(): as a call it took the caller's Steer by reference, which put
// that Steer on the stack (cfg 3: 28.94 ms inlined, 38.91 ms as a call).
__device__ __forceinline__ void steer_straight(const BikeParams &P, double ox, double oy, double theta, double gx, double gy, Steer &o) {
    double vx = gx - ox, vy = gy - oy;
    double nv = norm2(vx, vy);
    if (nv > 0.000001) {
        double sx = P.maxdrivedist * vx / nv, sy = P.maxdrivedist * vy / nv;
        if (norm2(sx, sy) > nv) {
        } else {
            gx = ox + sx;
            gy = oy + sy;
        }
    }
    o.x = gx; o.y = gy; o.theta = theta;
    o.steer = 0; o.iccx = o.iccy = o.rad = NAN; o.dist = 1; o.straight = true;
}

// rrt.py:306-524.  Inlined: one call site per kernel; as a call its Steer result travels through local memory
// (inlined 34.9 ms, as a call 36.2 ms on cfg 3).
__device__ __forceinline__ void steer(const BikeParams &P, double ox, double oy, double theta, double gx, double gy, double thetagoal, Steer &o) {
    double L = P.bikelength;
    double midx = 0.5 * (ox + gx), midy = 0.5 * (oy + gy);
    double bisx = ox - gx, bisy = oy - gy;
    double bfx, bfy, bnx, bny, pbx, pby;
    rotz(theta, L, 0.0, bfx, bfy);
    o.bfx = bfx; o.bfy = bfy;
    // r_90 (rrt.py:333-335,359) is a literal angle: matrix precomputed in P
    const double r00 = P.r90.m00, r01 = P.r90.m01, r10 = P.r90.m10;
    bnx = fma(r00, bfx, r01 * bfy); bny = fma(r10, bfx, r00 * bfy);
    pbx = fma(r00, bisx, r01 * bisy); pby = fma(r10, bisx, r00 * bisy);
    double a1, b1, c1, a2, b2, c2, ix, iy;
    linefrompoints(midx, midy, midx + pbx, midy + pby, a1, b1, c1);
    linefrompoints(ox, oy, ox + bnx, oy + bny, a2, b2, c2);
    if (!solve2(a1, b1, a2, b2, c1, c2, ix, iy) || cond2(a1, b1, a2, b2) > 1000000) {
        steer_straight(P, ox, oy, theta, gx, gy, o);
        return;
    }
    double rad = norm2(ox - ix, oy - iy);
    double pvx = bfx + ox, pvy = bfy + oy;
    double svx, svy;
    {
        double tx = pvx - ix, ty = pvy - iy;
        svx = fma(r00, tx, r01 * ty); svy = fma(r10, tx, r00 * ty);
    }
    double steerangle = standardangle(-anglebetween(bfx, bfy, svx, svy));
    bool point_to_goal_only = false;
    if (P.forwardonly && (steerangle > 90 || steerangle < -90)) {
        steerangle = steerangle + 180;
        steerangle = standardangle(steerangle);
    }
    if (steerangle < P.leftconstraint || steerangle > P.rightconstraint) {
        double fnx = 0, fny = 0;
        if (steerangle < P.leftconstraint) { steerangle = P.leftconstraint; rot_apply(P.rleft, bnx, bny, fnx, fny); }
        if (steerangle > P.rightconstraint) { steerangle = P.rightconstraint; rot_apply(P.rright, bnx, bny, fnx, fny); }
        linefrompoints(pvx, pvy, pvx + fnx, pvy + fny, a1, b1, c1);
        linefrompoints(ox, oy, ox + bnx, oy + bny, a2, b2, c2);
        if (!solve2(a1, b1, a2, b2, c1, c2, ix, iy) || cond2(a1, b1, a2, b2) > 1000000) {
            steer_straight(P, ox, oy, theta, gx, gy, o);
            return;
        }
        rad = norm2(ox - ix, oy - iy);
        point_to_goal_only = true;
    }
    double c_ccw;
    if ((steerangle >= 0 && steerangle < 90) || (steerangle <= -90 && steerangle > -180)) c_ccw = -90;
    else c_ccw = 90;
    double fvx, fvy;
    const Rot &rmc = (c_ccw < 0) ? P.r90 : P.rm90; // from_euler('z', -c_ccw): -c_ccw is exactly +90 or -90
    rot_apply(rmc, gx - ix, gy - iy, fvx, fvy);
    double final_angle = -anglebetween(1, 0, fvx, fvy);
    double mix_angle = P.weightxy * standardangle(final_angle) + (1 - P.weightxy) * standardangle(thetagoal);
    if (point_to_goal_only) mix_angle = anglebetween(1, 0, gx - ox, gy - oy);
    double thetagoal2 = mix_angle + c_ccw;
    double m1x, m1y, m2x, m2y;
    rotz(thetagoal2, 1.0, 0.0, m1x, m1y);
    {
        double n = norm2(m1x, m1y);
        m1x = rad * m1x / n; m1y = rad * m1y / n;
    }
    m1x = ix + m1x; m1y = iy + m1y;
    double thetagoal3 = thetagoal2 + 180;
    rotz(thetagoal3, 1.0, 0.0, m2x, m2y);
    {
        double n = norm2(m2x, m2y);
        m2x = rad * m2x / n; m2y = rad * m2y / n;
    }
    m2x = ix + m2x; m2y = iy + m2y;
    double ang_goal = anglebetween(1, 0, gx - ix, gy - iy);
    double diff1, diff2;
    {   // anglediff(a, ang_goal) twice (rrt.py:435-436): the quaternion of ang_goal is the same both times
        double sg, cg, s1, c1;
        quat_z(ang_goal, sg, cg);
        quat_z(anglebetween(1, 0, m1x - ix, m1y - iy), s1, c1);
        diff1 = anglediff_q(s1, c1, sg, cg);
        quat_z(anglebetween(1, 0, m2x - ix, m2y - iy), s1, c1);
        diff2 = anglediff_q(s1, c1, sg, cg);
    }
    final_angle = mix_angle;
    double gpx, gpy;
    if (fabs(diff1) < fabs(diff2)) { gpx = m1x; gpy = m1y; }
    else { gpx = m2x; gpy = m2y; final_angle = standardangle(final_angle - 180); }
    if (point_to_goal_only) {
        gpx = m1x; gpy = m1y;
        rot_apply(rmc, gpx - ix, gpy - iy, fvx, fvy);
        final_angle = -anglebetween(1, 0, fvx, fvy);
    }
    double iox = ox - ix, ioy = oy - iy;
    double angle = anglebetween(1, 0, gpx - ix, gpy - iy);
    double angle2 = anglebetween(1, 0, iox, ioy);
    double arcangle = anglediff(angle, angle2);
    if (steerangle > 0) { if (arcangle < 0) arcangle = 360 + arcangle; }
    else { if (arcangle > 0) arcangle = 360 - arcangle; }
    double traveldist = angle_to_arclength(rad, fabs(arcangle));
    if (traveldist > P.maxdrivedist) {
        traveldist = P.maxdrivedist;
        double mda = arclength_to_angle(rad, P.maxdrivedist);
        double rx, ry;
        if (steerangle < 0) rotz(-mda, iox, ioy, rx, ry);
        else rotz(mda, iox, ioy, rx, ry);
        gpx = rx + ix; gpy = ry + iy;
        rot_apply(rmc, gpx - ix, gpy - iy, fvx, fvy);
        final_angle = -anglebetween(1, 0, fvx, fvy);
    }
    o.x = gpx; o.y = gpy; o.theta = final_angle;
    o.steer = steerangle; o.iccx = ix; o.iccy = iy; o.rad = rad; o.dist = traveldist; o.straight = false;
}

// rrt.py:272-304 (dist = u[3], already divided by 3 by the caller, rrt.py:170)
// bf = Rz(theta)*[bikelength,0] as computed by steer() for the same origin bike (rrt.py:277-279 recomputes it)
// A call (the re-drive is the rarer branch of the expansion) whose pose comes back by value, in registers: through
// reference parameters it came back through the caller's stack.
struct Pose {
    double x, y, theta;
};
__device__ __noinline__ Pose drive_bf(const BikeParams &P, double ox, double oy, double bfx, double bfy, double usteer, double iccx,
                                      double iccy, double rad, double dist) {
    double angle = arclength_to_angle(rad, dist);
    double b1x, b1y;
    rot_apply(P.r180, bfx, bfy, b1x, b1y);
    bfx = (ox - iccx) + bfx; bfy = (oy - iccy) + bfy;
    b1x = (ox - iccx) + b1x; b1y = (oy - iccy) + b1y;
    double ra = (usteer < 0) ? -angle : angle;
    double tx, ty;
    Rot R = rot_make(ra); // the reference applies the same rotation to both points (rrt.py:293-294)
    rot_apply(R, bfx, bfy, tx, ty); bfx = tx; bfy = ty;
    rot_apply(R, b1x, b1y, tx, ty); b1x = tx; b1y = ty;
    bfx = iccx + bfx; bfy = iccy + bfy;
    b1x = iccx + b1x; b1y = iccy + b1y;
    double px = 0.5 * (b1x + bfx), py = 0.5 * (b1y + bfy);
    Pose f;
    f.theta = -anglebetween(1, 0, bfx - px, bfy - py);
    f.x = px; f.y = py;
    return f;
}
// rrt.py:272-304 from scratch (single-step entry point)
__device__ __forceinline__ void drive(const BikeParams &P, double ox, double oy, double theta, double usteer, double iccx, double iccy,
                                      double rad, double dist, double &fx, double &fy, double &fang) {
    double bfx, bfy;
    rotz(theta, P.bikelength, 0.0, bfx, bfy);
    const Pose f = drive_bf(P, ox, oy, bfx, bfy, usteer, iccx, iccy, rad, dist);
    fx = f.x; fy = f.y; fang = f.theta;
}

// Python round(): half to even
__device__ __forceinline__ long long py_round(double v) { return (long long)rint(v); }

// ---------------------------------------------------------------------------
// Midpoint-circle raster of search.getCircle (search.py:107-142) in closed
// form.  The loop emits, for y = 0..t_max, the 8 reflections of (x_y, y) where
//     x_y   = largest x with x*x - x < r*r - y*y           (decision variable)
//     t_max = largest t with 2*t*t + t < r*r                 (loop runs while x > y)
// (DESIGN.md has the derivation; tests compare against the literal loop for
// every r <= 2000).  Pixels outside the image are dropped (search.py:103).
// ---------------------------------------------------------------------------
__device__ __noinline__ long long circle_x(long long r, long long t) {
    // largest x >= 0 with x*(x-1) < c, c = r*r - t*t > 0
    long long c = r * r - t * t;
    long long x = (long long)((1.0 + sqrt(1.0 + 4.0 * (double)c)) * 0.5);
    while (x * (x - 1) >= c) --x;
    while ((x + 1) * x < c) ++x;
    return x;
}
__device__ __noinline__ long long circle_tmax(long long r) {
    // largest t >= 0 with 2*t*t + t < r*r; -1 when r == 0
    if (r <= 0) return -1;
    long long rr = r * r;
    long long t = (long long)((double)r * 0.70710678118654752440);
    while (t > 0 && 2 * t * t + t >= rr) --t;
    while (2 * (t + 1) * (t + 1) + (t + 1) < rr) ++t;
    return t;
}
// is offset (a, b) from the centre one of the raster pixels?
__device__ __noinline__ bool circle_member(long long r, long long a, long long b) {
    long long p = a < 0 ? -a : a, q = b < 0 ? -b : b;
    if (p < q) { long long t = p; p = q; q = t; }
    if (p == q) return false; // never emitted (search.py:100 / loop condition)
    if (q >= r) return false;
    return circle_x(r, q) == p;
}

struct ArcTest {
    // inputs of search.getArc (search.py:144-182) for the non-straight case
    double iccx, iccy, usteer;
    double u1x, u1y, u2x, u2y, n1, n2; // begin - icc, land - icc and their squared lengths
    int diff_lt_180;       // -1 unknown, else the outcome of `diff < 180` (search.py:170)
    bool ready;
};

// The reference keeps a circle pixel when the wrapped angle differences `forwardofbegin` and
// `backwardofgoal` (search.py:163-179) are >= 0.  With a = atan2(-vy, vx) the angle of a vector v
// (rrt.anglebetween([1,0], v)), the wrapped difference a2 - a1 in (-180, 180] is >= 0 exactly when
// sin(a2 - a1) = (v2x*v1y - v2y*v1x) / (|v1||v2|) >= 0.  The literal path (atan2, half-angle
// quaternions, atan2 again) carries ~1e-13 degrees of rounding noise, so whenever |sin| > 1e-9 the sign
// of the cross product IS the literal outcome and the three atan2 + sin/cos evaluations per blocked
// pixel are skipped; anything closer to 0 or 180 degrees goes through the literal computation.
#define TRRT_ARC_GUARD2 1e-18 /* (1e-9)^2, compared against cross^2 / (|v1|^2 |v2|^2) */

__device__ __forceinline__ int cross_sign(double v2x, double v2y, double v1x, double v1y, double n1n2) {
    // +1 / -1 when sin(a2 - a1) is safely positive / negative, 0 when too close to call
    double c = v2x * v1y - v2y * v1x;
    if (!(c * c > TRRT_ARC_GUARD2 * n1n2)) return 0;
    return c > 0 ? 1 : -1;
}

// The literal path (search.py:161-170).  Real calls, rare (|sin| <= 1e-9), that take the arc's vectors by value: a reference
// to the caller's ArcTest would put it on the stack.  Each call recomputes the begin / end quaternions from (u1, u2).
// `diff < 180` (search.py:170), the wrapped (endangle - beginangle) for a left turn, (beginangle - endangle) otherwise
__device__ __noinline__ int arc_literal_diff_lt180(double u1x, double u1y, double u2x, double u2y, double usteer) {
    double sb, cb, se, ce;
    quat_z(anglebetween(1, 0, u1x, u1y), sb, cb);
    quat_z(anglebetween(1, 0, u2x, u2y), se, ce);
    double d = (usteer < 0) ? anglediff_q(sb, cb, se, ce) : anglediff_q(se, ce, sb, cb);
    if (d < 0) d = 360 + d;
    return d < 180 ? 1 : 0;
}
// one of the two per-pixel differences (which: 0 = forwardofbegin, 1 = backwardofgoal) is >= 0
__device__ __noinline__ bool arc_literal_ge0(double u1x, double u1y, double u2x, double u2y, double usteer, double vx, double vy, int which) {
    double sb, cb, se, ce, sp, cp;
    quat_z(anglebetween(1, 0, u1x, u1y), sb, cb);
    quat_z(anglebetween(1, 0, u2x, u2y), se, ce);
    quat_z(anglebetween(1, 0, vx, vy), sp, cp);
    double d;
    if (usteer > 0) d = (which == 0) ? anglediff_q(sp, cp, sb, cb) : anglediff_q(se, ce, sp, cp);
    else d = (which == 0) ? anglediff_q(sb, cb, sp, cp) : anglediff_q(sp, cp, se, ce);
    return d >= 0;
}

// does getArc keep circle pixel (px, py)?  search.py:161-181.  Inlined: the cross products are a few dozen instructions, and
// as a call its ArcTest was on the stack of every raster (cfg 3: 28.94 ms inlined, 31.37 ms as a call).
__device__ __forceinline__ bool arc_keeps_pixel(ArcTest &A, double bx, double by, double lx, double ly, long long px, long long py) {
    if (!A.ready) { // lazily: only needed once a blocked circle pixel is met
        A.u1x = bx - A.iccx; A.u1y = by - A.iccy;
        A.u2x = lx - A.iccx; A.u2y = ly - A.iccy;
        A.n1 = A.u1x * A.u1x + A.u1y * A.u1y;
        A.n2 = A.u2x * A.u2x + A.u2y * A.u2y;
        // diff = wrapped (endangle - beginangle) for a left turn, (beginangle - endangle) otherwise, in [0, 360)
        int sd = (A.usteer < 0) ? cross_sign(A.u2x, A.u2y, A.u1x, A.u1y, A.n1 * A.n2) : cross_sign(A.u1x, A.u1y, A.u2x, A.u2y, A.n1 * A.n2);
        A.diff_lt_180 = (sd == 0) ? -1 : (sd > 0 ? 1 : 0);
        A.ready = true;
    }
    const double vx = (double)px - A.iccx, vy = (double)py - A.iccy;
    const double nv = vx * vx + vy * vy;
    int sf, sb;
    if (A.usteer > 0) { // forwardofbegin = begin - px, backwardofgoal = px - end
        sf = cross_sign(A.u1x, A.u1y, vx, vy, A.n1 * nv);
        sb = cross_sign(vx, vy, A.u2x, A.u2y, A.n2 * nv);
    } else {            // forwardofbegin = px - begin, backwardofgoal = end - px
        sf = cross_sign(vx, vy, A.u1x, A.u1y, A.n1 * nv);
        sb = cross_sign(A.u2x, A.u2y, vx, vy, A.n2 * nv);
    }
    const bool fob = (sf != 0) ? (sf > 0) : arc_literal_ge0(A.u1x, A.u1y, A.u2x, A.u2y, A.usteer, vx, vy, 0);
    const bool bog = (sb != 0) ? (sb > 0) : arc_literal_ge0(A.u1x, A.u1y, A.u2x, A.u2y, A.usteer, vx, vy, 1);
    if (A.diff_lt_180 < 0) A.diff_lt_180 = arc_literal_diff_lt180(A.u1x, A.u1y, A.u2x, A.u2y, A.usteer);
    if (A.diff_lt_180) return fob && bog;
    return fob || bog;
}

// rrt.py:173-174 for a curved edge: is any pixel of getArc(begin, land, u) not free?
// Candidate circle pixels are enumerated lane-parallel; only blocked in-bounds
// pixels pay for the angular test (free pixels cannot change the answer).
// T = int when the radius fits 15 bits (almost always), long long otherwise.
template <int G, typename T>
__device__ __noinline__ bool arc_blocked_impl(const Group<G> &g, const Grid &m, double bx, double by, double lx, double ly, double usteer,
                                              double iccx, double iccy, long long xc_, long long yc_, long long r_,
                                              unsigned long long *cand_px, unsigned long long *angle_tests) {
    const T r = (T)r_;
    // centres far outside the image cannot reach it with a small radius; clamp so that T never overflows
    const long long lim = (long long)1 << 20;
    const T xc = (T)(sizeof(T) == 4 ? (xc_ > lim ? lim : (xc_ < -lim ? -lim : xc_)) : xc_);
    const T yc = (T)(sizeof(T) == 4 ? (yc_ > lim ? lim : (yc_ < -lim ? -lim : yc_)) : yc_);
    ArcTest A;
    A.iccx = iccx; A.iccy = iccy; A.usteer = usteer; A.ready = false;
    bool hit = false;
    const T tmax = (T)circle_tmax(r_);
    const T rr = r * r;
    // Row ranges t for which a reflection can fall inside the image:
    //   kind 0: (xc +- x_t, yc + t)   kind 1: (xc +- x_t, yc - t)
    //   kind 2: (xc + t, yc +- x_t)   kind 3: (xc - t, yc +- x_t)
    T lo[4], hi[4];
    lo[0] = -yc;                 hi[0] = (T)m.W - 1 - yc; // valid(): y < shape[1]
    lo[1] = yc - ((T)m.W - 1);   hi[1] = yc;
    lo[2] = -xc;                 hi[2] = (T)m.H - 1 - xc; // valid(): x < shape[0]
    lo[3] = xc - ((T)m.H - 1);   hi[3] = xc;
#pragma unroll 1
    for (int k = 0; k < 4; k++) {
        T a = lo[k] < 0 ? 0 : lo[k], b = hi[k] > tmax ? tmax : hi[k];
        if (b < a) continue;
        T count = (b - a + 1) * 2; // two mirror pixels per row
        if (cand_px && g.gl == 0) *cand_px += (unsigned long long)count;
        T xt = -1; // x of the previous row handled by this lane (rows only grow, x only shrinks)
        for (T base = 0; base < count; base += G) {
            T j = base + g.gl;
            bool bad = false;
            if (j < count) {
                T t = a + (j >> 1);
                T c = rr - t * t;
                if (xt < 0) xt = (t == 0) ? r : (T)circle_x(r_, (long long)t); // x_0 = r
                while (xt * (xt - 1) >= c) --xt;
                T sx = (j & 1) ? -xt : xt;
                T px, py;
                if (k == 0) { px = xc + sx; py = yc + t; }
                else if (k == 1) { px = xc + sx; py = yc - t; }
                else if (k == 2) { px = xc + t; py = yc + sx; }
                else { px = xc - t; py = yc + sx; }
                if (px >= 0 && py >= 0 && px < (T)m.H && py < (T)m.W && !m.free_nb((int)px, (int)py)) {
                    if (angle_tests) *angle_tests += 1;
                    bad = arc_keeps_pixel(A, bx, by, lx, ly, (long long)px, (long long)py);
                }
            }
            if (g.any(bad)) { hit = true; break; }
        }
        if (hit) break;
    }
    if (hit) return true;
    // diagonal-gap pixels (search.py:124-138): added when none of the 4-neighbours of
    // (xc+rnd, yc+rnd) is an emitted (in-bounds) raster pixel
    long long rnd = py_round((double)r_ * 0.5 * sqrt(2.0));
    bool drawmore = true;
    {
        const int nx[4] = {1, -1, 0, 0}, ny[4] = {0, 0, 1, -1};
#pragma unroll
        for (int i = 0; i < 4; i++) {
            long long a = rnd + nx[i], b = rnd + ny[i];
            if (m.inb(xc_ + a, yc_ + b) && circle_member(r_, a, b)) drawmore = false;
        }
    }
    if (drawmore) {
        bool bad = false;
        for (int i = g.gl; i < 4; i += G) { // (+,+) (-,-) (+,-) (-,+)
            long long px = xc_ + ((i == 0 || i == 2) ? rnd : -rnd);
            long long py = yc_ + ((i == 0 || i == 3) ? rnd : -rnd);
            if (m.inb(px, py) && !m.free_nb((int)px, (int)py)) {
                if (angle_tests) *angle_tests += 1;
                bad = bad || arc_keeps_pixel(A, bx, by, lx, ly, px, py);
            }
        }
        if (g.any(bad)) return true;
    }
    return false;
}

// The generic raster (cooperative schedule, single-step kernel, enormous radii): a lane alone runs the 32-bit version
// when the radius allows, groups run the 64-bit version.  The speculative schedule uses arc_blocked_lane (trrt_lane.cuh).
template <int G>
__device__ __forceinline__ bool arc_blocked(const Group<G> &g, const Grid &m, double bx, double by, double lx, double ly,
                                            double usteer, double iccx, double iccy, double rad,
                                            unsigned long long *cand_px, unsigned long long *angle_tests) {
    long long xc = trunc_ll(iccx), yc = trunc_ll(iccy), r = trunc_ll(rad);
    if (G == 1 && r < 32768)
        return arc_blocked_impl<G, int>(g, m, bx, by, lx, ly, usteer, iccx, iccy, xc, yc, r, cand_px, angle_tests);
    return arc_blocked_impl<G, long long>(g, m, bx, by, lx, ly, usteer, iccx, iccy, xc, yc, r, cand_px, angle_tests);
}

} // namespace trrt
