/*
 * legacy_normals.c -- sequential CPU restatement of the device generator of
 * theta_rrt_b200/csrc/trrt_rng.cuh: numpy's legacy
 * RandomState(seed).standard_normal(n) (init_genrand seeding, MT19937,
 * legacy_double, the polar method of legacy_gauss), with log(r2) taken from
 * tl_log_dd (trrt_libm.h) when tl_log_decided settles it and from the host's
 * libm otherwise -- the same split the device makes.
 *
 * TEST INFRASTRUCTURE ONLY (tests/test_legacy_normals.py); the product never
 * loads it.  Built by oracle/legacy_normals.py with the flags of
 * oracle/Makefile.
 */
#include <math.h>
#include <stdint.h>

#include "../theta_rrt_b200/csrc/trrt_libm.h"

#define MT_N 624
#define MT_M 397

typedef struct {
    uint32_t key[MT_N];
    int pos;
} orc_mt;

void orc_init_genrand(uint32_t seed, uint32_t *key) {
    key[0] = seed;
    for (int i = 1; i < MT_N; i++) key[i] = 1812433253u * (key[i - 1] ^ (key[i - 1] >> 30)) + (uint32_t)i;
}

static void mt_gen(orc_mt *s) {
    uint32_t *k = s->key, y;
    int i;
    for (i = 0; i < MT_N - MT_M; i++) {
        y = (k[i] & 0x80000000u) | (k[i + 1] & 0x7fffffffu);
        k[i] = k[i + MT_M] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
    }
    for (; i < MT_N - 1; i++) {
        y = (k[i] & 0x80000000u) | (k[i + 1] & 0x7fffffffu);
        k[i] = k[i + (MT_M - MT_N)] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
    }
    y = (k[MT_N - 1] & 0x80000000u) | (k[0] & 0x7fffffffu);
    k[MT_N - 1] = k[MT_M - 1] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
    s->pos = 0;
}

static uint32_t mt_next(orc_mt *s) {
    if (s->pos == MT_N) mt_gen(s);
    uint32_t y = s->key[s->pos++];
    y ^= y >> 11;
    y ^= (y << 7) & 0x9d2c5680u;
    y ^= (y << 15) & 0xefc60000u;
    y ^= y >> 18;
    return y;
}

static double mt_double(orc_mt *s) {
    const int32_t a = (int32_t)(mt_next(s) >> 5), b = (int32_t)(mt_next(s) >> 6);
    return (a * 67108864.0 + b) / 9007199254740992.0;
}

/* out[0..n) = RandomState(seed).standard_normal(n).  stats[0] += logs evaluated, stats[1] += undecided ones (libm),
   stats[2] += decided ones whose tl_log_dd value differs from libm's log (must stay 0). */
void orc_legacy_normals(uint32_t seed, int64_t n, double *out, int64_t *stats) {
    orc_mt s;
    orc_init_genrand(seed, s.key);
    s.pos = MT_N;
    for (int64_t i = 0; i < n;) {
        double x1, x2, r2;
        do {
            x1 = 2.0 * mt_double(&s) - 1.0;
            x2 = 2.0 * mt_double(&s) - 1.0;
            r2 = x1 * x1 + x2 * x2;
        } while (r2 >= 1.0 || r2 == 0.0);
        double hi, lo, lg;
        tl_log_dd(r2, &hi, &lo);
        const double g = log(r2);
        stats[0]++;
        if (tl_log_decided(hi, lo)) {
            lg = hi;
            if (hi != g) stats[2]++;
        } else {
            lg = g;
            stats[1]++;
        }
        const double f = sqrt(-2.0 * lg / r2);
        out[i++] = f * x2;
        if (i < n) out[i++] = f * x1;
    }
}

/* tl_log_dd and tl_log_decided for an array */
void orc_tl_log_dd_array(const double *x, int64_t n, double *hi, double *lo, uint8_t *decided) {
    for (int64_t i = 0; i < n; i++) {
        tl_log_dd(x[i], &hi[i], &lo[i]);
        decided[i] = (uint8_t)tl_log_decided(hi[i], lo[i]);
    }
}
