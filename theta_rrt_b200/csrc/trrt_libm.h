/*
 * trrt_libm.h -- deterministic fp64 sin/cos/atan2 built only from IEEE-754
 * basic operations (+ - * / fma, rint, fabs), and the double-double log of
 * the seeded normal streams (tl_log_dd, at the end).
 *
 * Why this exists: the reference (rrt.py) routes every rotation and angle
 * through libm sin/cos/atan2 (via scipy Rotation and numpy).  CUDA's built-in
 * sin/cos/atan2 differ from glibc's in the last bit for a few percent of
 * arguments, and theta-rrt's tree growth amplifies such differences by ~10x per
 * tree level (tight 65-degree arcs), so two libms diverge into different trees
 * after a few thousand iterations.  Compiling ONE implementation for both the
 * host (gcc, -ffp-contract=off) and the device (nvcc, -fmad=false) makes host
 * and device results bit-identical, so the CUDA path can be checked against the
 * CPU oracle bit-for-bit at any tree size.
 *
 * Algorithms (published, restated here): Cody-Waite three-stage reduction by
 * pi/2 with 33-bit constant pieces, minimax kernels for sin/cos on
 * [-pi/4, pi/4] carrying the reduction tail (Sun fdlibm's published
 * coefficients), and atan2 by angle-addition against the breakpoints
 * {0, 1/2, 1, 3/2, inf} so only one division is needed.  Measured accuracy
 * against glibc 2.39 (tests/test_libm.py): max error < 1 ulp, bitwise equal to
 * glibc for >99% of arguments in the ranges the planner uses.  Accurate range
 * reduction holds for |x| < 2^20 * pi/2 (~1.6e6 rad); beyond that the result is
 * still deterministic but loses accuracy (no planner input gets there).
 */
#ifndef TRRT_LIBM_H
#define TRRT_LIBM_H

#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define TL_FN __host__ __device__ __forceinline__
/* the two entry points are real functions on the device: one copy each keeps the kernels' code
   footprint inside the instruction cache (inlining them at ~40 call sites made a 380 KB kernel
   that stalled 93% of the time on instruction fetch) */
#define TL_ENTRY static __host__ __device__ __noinline__
#else
#define TL_FN static inline
#define TL_ENTRY static inline
#endif

#define TL_PI 3.141592653589793116       /* np.pi */
#define TL_PI_LO 1.2246467991473531772e-16 /* pi - TL_PI */
#define TL_PIO2 1.570796326794896558
#define TL_PIO2_LO 6.123233995736765886e-17

/* sin on [-pi/4, pi/4], x + y is the reduced argument (y = tail).
   Polynomials are evaluated with explicit fma() (Horner): same bits on host and device, half the
   instructions of separate multiply/add. */
TL_FN double tl_ksin(double x, double y) {
    const double S1 = -1.66666666666666324348e-01, S2 = 8.33333333332248946124e-03,
                 S3 = -1.98412698298579493134e-04, S4 = 2.75573137070700676789e-06,
                 S5 = -2.50507602534068634195e-08, S6 = 1.58969099521155010221e-10;
    double z = x * x;
    double zl = fma(x, x, -z);                 /* x*x = z + zl exactly */
    double v = z * x;
    double vl = fma(x, zl, fma(z, x, -v));     /* x^3 = v + vl (to ~2^-106) */
    double r = fma(z, fma(z, fma(z, fma(z, S6, S5), S4), S3), S2);
    double t1 = S1 * v;                        /* leading correction -x^3/6 */
    double t1l = fma(S1, vl, fma(S1, v, -t1));
    /* tail terms: y*(1 - z/2) + x^5 * r */
    double small = fma(-z, fma(-v, r, 0.5 * y), y) + t1l;
    double s = x + t1;                         /* |x| >= |t1| : Fast2Sum */
    double se = t1 - (s - x);
    return s + (se + small);
}

/* cos on [-pi/4, pi/4] */
TL_FN double tl_kcos(double x, double y) {
    const double C1 = 4.16666666666666019037e-02, C2 = -1.38888888888741095749e-03,
                 C3 = 2.48015872894767294178e-05, C4 = -2.75573143513906633035e-07,
                 C5 = 2.08757232129817482790e-09, C6 = -1.13596475577881948265e-11;
    double z = x * x;
    double zl = fma(x, x, -z);
    double r = z * fma(z, fma(z, fma(z, fma(z, fma(z, C6, C5), C4), C3), C2), C1);
    double hz = 0.5 * z;
    double w = 1.0 - hz;
    double tail = fma(z, r, -fma(x, y, 0.5 * zl));
    return w + (((1.0 - w) - hz) + tail);      /* 1 - hz carried exactly as w + ((1-w)-hz) */
}

/* reduce x to y0 + y1 in [-pi/4, pi/4], return quadrant (mod 4 meaningful) */
TL_FN int tl_rem_pio2(double x, double *y0, double *y1) {
    const double INVPIO2 = 6.36619772367581382433e-01;
    const double P1 = 1.57079632673412561417e+00, P1T = 6.07710050650619224932e-11;
    const double P2 = 6.07710050630396597660e-11, P2T = 2.02226624879595063154e-21;
    const double P3 = 2.02226624871116645580e-21, P3T = 8.47842766036889956997e-32;
    double fn = rint(x * INVPIO2);
    double r = fma(-fn, P1, x); /* fn*P1 is exact for |fn| < 2^20 (P1 has 33 bits), so this is x - fn*P1 */
    double w = fn * P1T;
    double y = r - w;
    /* cancellation check: redo with more bits of pi/2 when the result is small */
    if (fabs(y) < fabs(x) * 1.52587890625e-05 /* 2^-16 */) {
        double t = r;
        w = fn * P2;
        r = t - w;
        w = fn * P2T - ((t - r) - w);
        y = r - w;
        if (fabs(y) < fabs(x) * 1.7763568394002505e-15 /* 2^-49 */) {
            t = r;
            w = fn * P3;
            r = t - w;
            w = fn * P3T - ((t - r) - w);
            y = r - w;
        }
    }
    *y0 = y;
    *y1 = (r - y) - w;
    /* fn is integral and |fn| < 2^31 for every finite planner input */
    return (int)((long long)fn & 3);
}

TL_FN void tl_sincos_body(double x, double *s, double *c) {
    double ax = fabs(x);
    double y0, y1;
    if (!(ax < 1.0e300)) { /* inf / nan / absurd */
        *s = x - x; *c = x - x; return;
    }
    if (ax < 7.450580596923828125e-09 /* 2^-27 */) { *s = x; *c = 1.0; return; }
    /* below pi/4 the reduction is the identity (fn = 0: y0 = x, y1 = +0, n = 0), so it runs unconditionally and the
       lanes of a warp do not split on the size of their argument */
    const int n = tl_rem_pio2(x, &y0, &y1);
    double ks = tl_ksin(y0, y1), kc = tl_kcos(y0, y1);
    double ss = (n & 1) ? kc : ks, cc = (n & 1) ? ks : kc;
    /* quadrant signs: n=0 (s,c) n=1 (c,-s) n=2 (-s,-c) n=3 (-c,s) */
    *s = (n & 2) ? -ss : ss;
    *c = ((n + 1) & 2) ? -cc : cc;
}
TL_ENTRY void tl_sincos(double x, double *s, double *c) { tl_sincos_body(x, s, c); }
/* the same by value: on the device the two results come back in registers, where tl_sincos's pointers put the caller's
   s and c on its stack (cfg-3 RRT kernel: 28.94 ms, 29.18 ms through tl_sincos) */
typedef struct { double s, c; } tl_sc;
TL_ENTRY tl_sc tl_sincos_v(double x) {
    tl_sc r;
    tl_sincos_body(x, &r.s, &r.c);
    return r;
}

/* odd minimax polynomial for atan(t) - t on |t| <= 7/16 (fdlibm aT[]) */
TL_FN double tl_atan_poly(double t) {
    const double A0 = 3.33333333333329318027e-01, A1 = -1.99999999998764832476e-01,
                 A2 = 1.42857142725034663711e-01, A3 = -1.11111104054623557880e-01,
                 A4 = 9.09088713343650656196e-02, A5 = -7.69187620504482999495e-02,
                 A6 = 6.66107313738753120669e-02, A7 = -5.83357013379057348645e-02,
                 A8 = 4.97687799461593236017e-02, A9 = -3.65315727442169155270e-02,
                 A10 = 1.62858201153657823623e-02;
    double z = t * t;
    double zl = fma(t, t, -z);
    double w = z * z;
    double s1 = z * fma(w, fma(w, fma(w, fma(w, fma(w, A10, A8), A6), A4), A2), A0);
    double s2 = w * fma(w, fma(w, fma(w, fma(w, A9, A7), A5), A3), A1);
    return t * fma(A0, zl, s1 + s2); /* atan(t) = t - this */
}

/* zeros, infinities, NaN: the values numpy / C99 define */
TL_FN double tl_atan2_special(double y, double x) {
    if (x != x || y != y) return x + y;
    double ay = fabs(y), ax = fabs(x);
    int yneg = signbit(y) ? 1 : 0, xneg = signbit(x) ? 1 : 0;
    if (ay == 0.0) { /* +-0 */
        if (xneg) return yneg ? -TL_PI : TL_PI;
        return y; /* +-0 */
    }
    if (ax == 0.0) return yneg ? -TL_PIO2 : TL_PIO2;
    if (isinf(ax)) {
        if (isinf(ay)) {
            double q = xneg ? 3.0 * 0.78539816339744827900 : 0.78539816339744827900;
            return yneg ? -q : q;
        }
        if (xneg) return yneg ? -TL_PI : TL_PI;
        return yneg ? -0.0 : 0.0;
    }
    return yneg ? -TL_PIO2 : TL_PIO2; /* |y| = inf, x finite */
}

TL_ENTRY double tl_atan2(double y, double x) {
    double ay = fabs(y), ax = fabs(x);
    /* one test for every special case: both magnitudes must be finite and non-zero */
    if (!(ax > 0.0 && ay > 0.0 && ax < INFINITY && ay < INFINITY)) return tl_atan2_special(y, x);
    /* first-quadrant angle a = atan(ay/ax) by angle addition against c in {0, 1/2, 1, 2, inf}:
       atan(ay/ax) = atan(c) + atan(t), t = (ay - c*ax)/(ax + c*ay), |t| <= 7/16.
       c*ax, c*ay and the numerator are exact (Sterbenz); the denominator is carried as dh + dl. */
    /* The octant is chosen with selects, not branches (lanes of a warp hold unrelated vectors): c = 0 and c = inf run
       through the general formula with c = 0 -- for c = inf on the swapped pair (-ax, ay) -- which reproduces
       num = ay (resp. -ax), dh = ax (resp. ay), dl = +0 exactly (0*v = +-0, v - 0 = v, v + +-0 = v). */
    const int c0 = ay * 16.0 < ax * 7.0;              /* ratio < 7/16: c = 0 */
    const int cinf = !c0 && (ay * 4.0 >= ax * 16.0);  /* ratio >= 4: c = inf, atan = pi/2 - atan(ax/ay) */
    const int chalf = ay * 16.0 < ax * 11.0, cone = ay * 2.0 < ax * 3.0;
    const double c = (c0 | cinf) ? 0.0 : (chalf ? 0.5 : (cone ? 1.0 : 2.0));
    const double hi = c0 ? 0.0 : (cinf ? 1.57079632679489655800e+00
                                       : (chalf ? 4.63647609000806093515e-01 : (cone ? 7.85398163397448278999e-01 : 1.10714871779409040897e+00)));
    const double lo = c0 ? 0.0 : (cinf ? 6.12323399573676603587e-17
                                       : (chalf ? 2.26987774529616870924e-17 : (cone ? 3.06161699786838301793e-17 : 9.40447137356637941245e-17)));
    const double yy = cinf ? -ax : ay, xx = cinf ? ay : ax;
    const double cx = c * xx, cy = c * yy;
    const double num = yy - cx;
    const double dh = xx + cy;
    const double bb = dh - xx;             /* TwoSum(xx, cy) */
    const double dl = (xx - (dh - bb)) + (cy - bb);
    /* one division: t approximates NUM/DEN, e is the remainder of the exact quotient */
    double rdh = 1.0 / dh;
    double t = num * rdh;
    double e = fma(-t, dl, fma(-t, dh, num)) * rdh; /* NUM/(dh+dl) = t + e */
    double p = tl_atan_poly(t);
    /* atan(t + e) ~= t - p + e*(1 - t*t) (|e| <= ~2 ulp(t), |t| <= 7/16) */
    double small = fma(e, fma(-t, t, 1.0), -p) + lo;
    /* first-quadrant result = s + rest, |rest| << |s|; with hi = 0 this is s = t, rest = small exactly */
    const double s = hi + t;                 /* |hi| >= |t| or hi = 0 : Fast2Sum */
    const double rest = (t - (s - hi)) + small;
    /* second/third quadrant: pi - (s + rest) with the low word of pi */
    const double u = TL_PI - s;              /* |pi| >= |s| : Fast2Sum */
    const double ue = (TL_PI - u) - s;
    const double r = (x > 0.0) ? s + rest : u + ((ue + TL_PI_LO) - rest);
    return (y < 0.0) ? -r : r;
}

/* ---------------------------------------------------------------------------
 * log(x) for x in (0, 1) as a double-double, and the test of whether glibc's
 * log must round it like correct rounding does.
 *
 * numpy's legacy polar method (legacy_gauss) calls the host libm's log, whose
 * results are not correctly rounded (glibc documents < 0.519 ulp).  The device
 * generator therefore settles only the values whose glibc rounding is forced:
 * if the exact log lies more than TL_LOG_MARGIN ulp + the error of tl_log_dd
 * away from every rounding midpoint, any result within 0.5 + 0.019 ulp of it
 * is the correctly rounded double, which is hi.  The rest ("undecided") are
 * handed to the host's libm.
 *
 * Algorithm: x = 2^k * m with m in [c, 2c), c = RN(sqrt(1/2)) (frexp, exact);
 * s = (m - 1) / (m + 1), |s| <= 0.17158; log(m) = 2s * F(t), t = s^2,
 * F(t) = 1 + t/3 + t^2/5 + ... ; log(x) = k*ln2 + log(m).
 * Error bound (relative to |log x|), derived:
 *   - m - 1 is exact (Sterbenz), m + 1 = dh + dl exactly (TwoSum); s = sh + sl
 *     from one division plus the exact fma remainder: |err| <= 2^-103 |s|.
 *   - t = s^2 in double-double: <= 2^-101 |t|.
 *   - F: 1, 1/3, 1/5 and the products with t in double-double (each step
 *     <= 2^-104 relative); R(t) = 1/7 + t/9 + ... + t^9/25 in double Horner
 *     with coefficients rounded to double: |R err| <= 2^-52, which enters F
 *     as t^3 |R err| <= 0.02944^3 * 2^-52 < 2^-67.2.  Truncation after the
 *     t^12/25 term: sum_{j>=13} t^j/(2j+1) <= t^13/27/(1-t) < 2^-70.8.
 *     F >= 1, so F carries < 2^-67.1 relative error.
 *   - log(m) = 2s * F, one double-double product: < 2^-67.0 relative.
 *   - k != 0 means x < c, m in [c, 2c): |log m| <= 0.3466 <= |k ln2| / 2, so
 *     |log x| >= |k ln2| / 2 >= |log m|; k*ln2 is formed from a 107-bit ln2
 *     with one exact product: the sum keeps < 2^-67 + 2^-103 relative.
 * TL_LOG_EPS = 2^-66 is the bound used (2x headroom over the derivation);
 * tests/test_legacy_normals.py checks it against decimal at 60 digits.
 * ------------------------------------------------------------------------- */
#define TL_LOG_EPS 1.3552527156068805e-20   /* 2^-66 */
#define TL_LOG_MARGIN 0.03125               /* 2^-5 ulp > glibc's 0.019-ulp excess over correct rounding */

TL_FN void tl_two_sum(double a, double b, double *s, double *e) {
    const double x = a + b, bb = x - a;
    *e = (a - (x - bb)) + (b - bb);
    *s = x;
}
TL_FN void tl_fast_two_sum(double a, double b, double *s, double *e) { /* |a| >= |b| or a = 0 */
    const double x = a + b;
    *e = b - (x - a);
    *s = x;
}
/* (ah + al) * (bh + bl), normalised */
TL_FN void tl_dd_mul(double ah, double al, double bh, double bl, double *ph, double *pl) {
    const double p = ah * bh;
    const double e = fma(ah, bh, -p) + fma(ah, bl, al * bh);
    tl_fast_two_sum(p, e, ph, pl);
}
/* (ah + al) + (bh + bl), normalised */
TL_FN void tl_dd_add(double ah, double al, double bh, double bl, double *sh, double *sl) {
    double s, e;
    tl_two_sum(ah, bh, &s, &e);
    e += al + bl;
    tl_fast_two_sum(s, e, sh, sl);
}

TL_ENTRY void tl_log_dd(double x, double *hi, double *lo) {
    int k;
    double m = frexp(x, &k); /* x = m * 2^k, m in [1/2, 1) */
    if (m < 0.7071067811865476) { m *= 2.0; k -= 1; }
    const double num = m - 1.0;
    double dh, dl;
    tl_two_sum(m, 1.0, &dh, &dl);
    const double sh = num / dh;
    const double sl = fma(-sh, dl, fma(-sh, dh, num)) / dh;
    double th, tl;
    tl_dd_mul(sh, sl, sh, sl, &th, &tl);
    /* R(t) = sum_{j=3..12} t^(j-3) / (2j+1) */
    double r = 1.0 / 25;
    r = fma(r, th, 1.0 / 23); r = fma(r, th, 1.0 / 21); r = fma(r, th, 1.0 / 19); r = fma(r, th, 1.0 / 17);
    r = fma(r, th, 1.0 / 15); r = fma(r, th, 1.0 / 13); r = fma(r, th, 1.0 / 11); r = fma(r, th, 1.0 / 9);
    r = fma(r, th, 1.0 / 7);
    double fh, fl;
    tl_dd_mul(th, tl, r, 0.0, &fh, &fl);
    tl_dd_add(0.2, -1.1102230246251566e-17, fh, fl, &fh, &fl);            /* 1/5 */
    tl_dd_mul(th, tl, fh, fl, &fh, &fl);
    tl_dd_add(0.3333333333333333, 1.850371707708594e-17, fh, fl, &fh, &fl); /* 1/3 */
    tl_dd_mul(th, tl, fh, fl, &fh, &fl);
    tl_dd_add(1.0, 0.0, fh, fl, &fh, &fl);
    double lh, ll;
    tl_dd_mul(2.0 * sh, 2.0 * sl, fh, fl, &lh, &ll);                         /* log(m) */
    if (k != 0) {
        const double L2H = 0.6931471805599453, L2L = 2.3190468138462996e-17; /* ln 2 */
        const double kd = (double)k;
        const double p = kd * L2H;
        const double pe = fma(kd, L2H, -p) + kd * L2L;
        tl_dd_add(p, pe, lh, ll, &lh, &ll);
    }
    *hi = lh;
    *lo = ll;
}

/* 1 when hi (= RN(hi + lo)) is the double that glibc's log returns: the exact value, within TL_LOG_EPS of hi + lo,
   is more than TL_LOG_MARGIN ulp away from the rounding midpoint on lo's side (the one on the other side is at
   least a quarter ulp away).  hi != 0. */
TL_FN int tl_log_decided(double hi, double lo) {
    const double ahi = fabs(hi);
    int e;
    const double f = frexp(ahi, &e);
    const double ulp = ldexp(1.0, e - 53);
    /* toward zero from a power of two the spacing of the doubles halves */
    const double side = (f == 0.5 && (lo < 0.0) != (hi < 0.0) && lo != 0.0) ? 0.5 * ulp : ulp;
    const double dist = 0.5 * side - fabs(lo);
    return dist > TL_LOG_MARGIN * ulp + 2.0 * TL_LOG_EPS * ahi;
}

#endif /* TRRT_LIBM_H */
