// trrt_los.cuh -- K4b: search.lineofsight (search.py:35-94) for independent segments over a STRIP copy of the
// occupancy grid, eight pixels of a ray per step, lanes picking up the next segment as soon as theirs is decided.
//
// Why a second layout.  In the row-major grid a 32-byte sector is 256 pixels of ONE row, so every pixel of a steep
// ray is a new sector and a new load (the one-thread-per-ray kernel sat at 62 % of the L1 sector throughput with 53
// sectors per ray).  Bresenham advances the driving axis by one per pixel and the other axis by at most one, so the
// eight pixels whose driving coordinate lies in one aligned block of 8 stay inside an 8 x 8 window in the direction of
// travel.  The strip copy stores, for every aligned block of 8 along the driving axis and every aligned offset 8K-8 on
// the other axis, the 8 x 16 pixels [8c, 8c+8) x [8K-8, 8K+8) as one 16-byte entry (byte j = the 8 pixels at offset
// 8K-8+j, bit i = driving coordinate 8c+i, 1 = free, outside the image 0).  Entries overlap by half, so the window of
// any block is inside ONE entry: one 16-byte load per lane and 8 pixels.  There are two orientations: 0 for rays
// driven by x (plotLineLow, search.py:58-75), 1 for rays driven by y (plotLineHigh, search.py:77-94), which is the
// same layout of the transposed image.  Per map: 2 * (tp+1) * tp entries, tp = ceil(side / 8) (4x the packed rows).
//
// A step of a lane (uniform control flow, no per-pixel branches):
//   1. load the entry of the block from (block index, other-axis coordinate at the block's first pixel);
//   2. the reference's running-error recurrence (D > 0 -> step, D -= 2*dmaj; D += 2*dmin) in closed form: the window
//      row of slot k is floor((u + k*2*dmin) / (2*dmaj)), u the phase of D at slot 0; the 8 quotients are exact
//      FFMA + magic-number roundings and land as nibbles of a PRMT selector;
//   3. shift the window to the entry's byte offset (funnel shift), gather the 8 rows with two PRMTs, and pick bit k of
//      row k with the diagonal masks 0x08040201 / 0x80402010 restricted to the pixels that belong to the segment.
// The first block starts at the aligned coordinate below the segment's first pixel, in the state the recurrence would
// have had klo pixels before the segment, so that it reaches the reference's D0 and coordinate exactly at slot klo.
//
// Why refill.  Rays differ wildly in length and 88 % of the cfg-4 rays are blocked after a few pixels; with one
// ray per thread a warp ran at 8 active lanes per instruction.  Here a warp owns a contiguous range of segments and
// hands the next ones to its idle lanes (ballot + prefix popcount) whenever at least `refill_min` lanes are idle.
//
// The result is the AND over the ray's pixels, so grouping the tests by blocks cannot change it; the pixel sequence
// is exactly the reference's after the canonicalisation of search.py:47-56.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace trrt {

// byte of packed row y holding pixels x = 8*xb .. 8*xb+7 (0 outside the image; padding bits of the rows are 0)
__device__ __forceinline__ unsigned strip_row_byte(const uint32_t *__restrict__ bits, int side, int wpr, int tp, int y, int xb) {
    if (y < 0 || y >= side || xb < 0 || xb >= tp) return 0u;
    return (__ldg(bits + (size_t)y * wpr + (xb >> 2)) >> ((xb & 3) * 8)) & 0xffu;
}

// Strip entry (K, c) of orientation `orient` of one map (src = its packed rows), built from the packed rows.  The one
// definition of the strip layout on the write side: the full build and the patch after a map edit both call it.
__device__ __forceinline__ uint4 strip_entry(const uint32_t *__restrict__ src, int side, int wpr, int tp, int orient, int K, int c) {
    unsigned w[4] = {0u, 0u, 0u, 0u};
    if (!orient) {
        // driving axis x: byte j = pixels (8c .. 8c+7, y = 8K-8+j)
#pragma unroll
        for (int j = 0; j < 16; j++) w[j >> 2] |= strip_row_byte(src, side, wpr, tp, 8 * K - 8 + j, c) << ((j & 3) * 8);
    } else {
        // driving axis y: byte j = pixels (x = 8K-8+j, 8c .. 8c+7): transpose 8 rows of 16 pixels
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const int y = 8 * c + i;
            const unsigned v = strip_row_byte(src, side, wpr, tp, y, K - 1) | (strip_row_byte(src, side, wpr, tp, y, K) << 8);
#pragma unroll
            for (int j = 0; j < 16; j++) w[j >> 2] |= ((v >> j) & 1u) << ((j & 3) * 8 + i);
        }
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
}

// bit-packed rows -> strip entries of both orientations; one thread per entry
__global__ void tile_grid_kernel(const uint32_t *__restrict__ bits, int n_maps, int side, int wpr, int tp, uint4 *__restrict__ tiles) {
    const size_t epo = (size_t)(tp + 1) * tp, total = epo * 2 * n_maps;
    for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
        const size_t m = e / (2 * epo), r = e - m * 2 * epo;
        const int orient = r >= epo, K = (int)((r - (orient ? epo : 0)) / tp), c = (int)((r - (orient ? epo : 0)) - (size_t)K * tp);
        tiles[e] = strip_entry(bits + m * (size_t)side * wpr, side, wpr, tp, orient, K, c);
    }
}

// Floor of a small quotient on the FMA pipe.  For integers 0 <= x < 2^20 and 0 < d < 2^16 with x / d < 16:
//     floor(x / d) = low bits of  fmaf(x, rcp, hrm) + 1.5 * 2^23,   rcp = rn(1 / d),  hrm = rn(0.5 * rcp - 0.5).
// (x + 0.5) / d is at least 0.5 / d >= 2^-17 away from every integer, the computed value is within 2^-19 of it
// (rcp and hrm are correctly rounded, the product is exact in the fma, |value| < 16), so after the shift by -0.5 the
// round-to-nearest of the magic addition is the floor.  tests/test_los_strip_model.py checks the formula against the
// integer division on the boundary cases (x a multiple of d, one below) up to d = 65534.
#define TRRT_LOS_MAGIC 12582912.0f   /* 1.5 * 2^23: float bits 0x4B400000 + n for the integer n it is added to */
#define TRRT_LOS_MAGIC_BITS 0x4B400000u

// One block of a ray: the 8 slots whose driving coordinate is A .. A+7 (A a multiple of 8), of which slots
// klo .. min(7, aend - A) belong to the segment.  b is the other-axis coordinate at slot 0 and u the phase of the
// reference's running error there, u = D - (2*dmin - 2*dmaj + 1) in [0, 2*dmaj): the recurrence of search.py:68-74 /
// :87-93 (D > 0 -> step, D -= 2*dmaj; D += 2*dmin) keeps D in (2*dmin - 2*dmaj, 2*dmin], so after k pixels
// u_k = (u + k*2*dmin) mod 2*dmaj and the number of steps taken is floor((u + k*2*dmin) / (2*dmaj)) (DESIGN.md 8.1).
// The 8 quotients come from the FMA pipe (see above) instead of 8 dependent compare / select / add triples on the
// integer pipe, which is the one this kernel saturates.  u is kept as a float (an exact integer < 2^17).
// gtn = base of the orientation, moved on by one row of entries when the ray travels towards larger coordinates (so
// that the entry index is (b >> 3) * tp + (A >> 3) either way).  b and u are advanced to slot 0 of the next block.
// Returns a non-zero word when one of the segment's pixels is blocked.
struct StripRay {
    float rcp, slope, hrm, d8, dmaj2; // 1 / (2*dmaj), 2*dmin / (2*dmaj), 0.5 * rcp - 0.5, 8 * 2*dmin, 2*dmaj
};
__device__ __forceinline__ void strip_ray_consts(StripRay &r, float dmaj2f, float d8f) {
    r.dmaj2 = dmaj2f; r.d8 = d8f;
    r.rcp = __frcp_rn(dmaj2f);
    r.slope = (d8f * 0.125f) * r.rcp;
    r.hrm = 0.5f * r.rcp - 0.5f;
}
__device__ __forceinline__ unsigned strip_block(const uint4 *__restrict__ gtn, int tp, int A, int aend, int klo, bool neg, const StripRay &r, int &b,
                                                float &u) {
    const uint4 wv = __ldg(gtn + ((b >> 3) * tp + (A >> 3)));
    const int sb = (b & 7) + (neg ? 1 : 0); // byte of the entry where the window starts
    const float base = fmaf(u, r.rcp, r.hrm);
    unsigned acc = 0; // nibble k = number of steps taken before slot k (slot 0: none)
#pragma unroll
    for (int k = 1; k < 8; k++) acc += __float_as_uint(fmaf(r.slope, (float)k, base) + TRRT_LOS_MAGIC) << (4 * k);
    unsigned sel = acc - 0xf4000000u; // the magic's exponent bits, summed over the seven shifts (mod 2^32)
    const float r8 = fmaf(r.slope, 8.0f, base) + TRRT_LOS_MAGIC;
    const int j = (int)(__float_as_uint(r8) - TRRT_LOS_MAGIC_BITS);
    u = fmaf(-(r8 - TRRT_LOS_MAGIC), r.dmaj2, u + r.d8); // exact: integers below 2^24
    b += neg ? -j : j;
    const int q = sb >> 2, sh = (sb & 3) * 8;
    const unsigned r0 = q == 0 ? wv.x : q == 1 ? wv.y : wv.z;
    const unsigned r1 = q == 0 ? wv.y : q == 1 ? wv.z : wv.w;
    const unsigned r2 = q == 0 ? wv.z : wv.w; // unused when q == 2 (sh == 0)
    const unsigned ulo = __funnelshift_r(r0, r1, sh), uhi = __funnelshift_r(r1, r2, sh);
    if (neg) sel ^= 0x77777777u; // travel towards smaller coordinates: row j is byte 7 - j
    const unsigned rows_lo = __byte_perm(ulo, uhi, sel & 0xffffu), rows_hi = __byte_perm(ulo, uhi, sel >> 16);
    const int left = aend - A, khi = left < 7 ? left : 7;
    const unsigned kmask = ((2u << khi) - 1u) & ~((1u << klo) - 1u);
    const unsigned rep = kmask * 0x01010101u;
    return (~rows_lo & rep & 0x08040201u) | (~rows_hi & rep & 0x80402010u);
}

constexpr int LOS_WARPS = 4, LOS_CTAS_PER_SM = 8; // CTA shape of los_tiled_kernel, also used by its launch
__global__ void __launch_bounds__(LOS_WARPS * 32, LOS_CTAS_PER_SM)
    los_tiled_kernel(const uint4 *__restrict__ tiles, int side, int tp, const int32_t *__restrict__ map_id, const int4 *__restrict__ seg, long long n,
                     int rays_per_warp, int refill_min, int coop_max, uint8_t *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const unsigned lt = (1u << lane) - 1u;
    const long long begin = ((blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5) * rays_per_warp;
    if (begin >= n) return;
    const int cnt = (int)((begin + rays_per_warp < n) ? rays_per_warp : n - begin); // segments of this warp
    seg += begin;
    out += begin;
    if (map_id) map_id += begin;
    const int epo = (tp + 1) * tp; // entries per orientation (< 2^25 for side <= 32768)
    int nxt = 0;                   // warp-uniform: first segment of the range not yet handed to a lane

    bool active = false, neg = false;
    const uint4 *gtn = tiles;
    int idx = 0, a = 0, aend = 0, b = 0, klo = 0;
    float u = 0.0f;
    StripRay R = {0.5f, 0.0f, -0.25f, 0.0f, 2.0f};

    for (;;) {
        unsigned act = __ballot_sync(0xffffffffu, active);
        int na = __popc(act);
        if (nxt < cnt && 32 - na >= refill_min) {
            if (!active) {
                const int i = nxt + __popc(~act & lt);
                if (i < cnt) {
                    const int4 s = __ldg(seg + i);
                    // search.valid on both endpoints (search.py:17-24, :36); maps are square
                    if ((unsigned)s.x < (unsigned)side && (unsigned)s.y < (unsigned)side && (unsigned)s.z < (unsigned)side &&
                        (unsigned)s.w < (unsigned)side) {
                        const bool low = abs(s.w - s.y) < abs(s.z - s.x); // search.py:47
                        int p0 = low ? s.x : s.y, q0 = low ? s.y : s.x, p1 = low ? s.z : s.w, q1 = low ? s.w : s.z;
                        if (p0 > p1) { int t = p0; p0 = p1; p1 = t; t = q0; q0 = q1; q1 = t; } // search.py:48-56
                        const int dmaj = p1 - p0, dq = q1 - q0;
                        neg = dq < 0;
                        const int dmaj2 = dmaj ? 2 * dmaj : 2, dmin2 = 2 * abs(dq); // a single pixel never steps
                        strip_ray_consts(R, (float)dmaj2, (float)(8 * dmin2));
                        klo = p0 & 7; a = p0 & ~7; aend = p1;
                        // The reference starts at D0 = 2*dmin - dmaj (search.py:66 / :85), i.e. phase dmaj - 1, at slot klo of
                        // the first block.  Slot 0 gets the state the recurrence would have had klo pixels earlier: phase
                        // (dmaj - 1 - klo*2*dmin) mod 2*dmaj and the other-axis coordinate that many steps back, so that
                        // the block step needs no special case (the slots before klo are masked).
                        const int w = (dmaj ? dmaj - 1 : 0) - klo * dmin2 + 7 * dmaj2; // >= 0
                        const int qd = (int)(__float_as_uint(fmaf((float)w, R.rcp, R.hrm) + TRRT_LOS_MAGIC) - TRRT_LOS_MAGIC_BITS); // w / dmaj2
                        u = (float)(w - qd * dmaj2);
                        b = q0 + (neg ? 7 - qd : qd - 7);
                        gtn = tiles + ((size_t)(map_id ? __ldg(map_id + i) : 0) * 2 * epo + (low ? 0 : epo) + (neg ? 0 : tp));
                        idx = i;
                        active = true;
                    } else {
                        out[i] = 0;
                    }
                }
            }
            nxt += 32 - na;
            act = __ballot_sync(0xffffffffu, active);
            na = __popc(act);
        }
        if (na == 0) {
            if (nxt >= cnt) break;
            continue;
        }
        if (nxt < cnt || na > coop_max) {
            // every lane advances its own ray by one block
            if (active) {
                const unsigned bad = strip_block(gtn, tp, a, aend, klo, neg, R, b, u);
                a += 8;
                klo = 0;
                if (bad != 0u || a > aend) {
                    out[idx] = bad ? 0 : 1;
                    active = false;
                }
            }
        } else {
            // The warp's range is used up and few rays are left: the idle lanes join in.  The lanes are split into
            // groups of G = 32 / nextpow2(na); group g takes the g-th remaining ray and member m its m-th next block,
            // whose phase and coordinate follow from the same modular rule, m blocks at once (integer division).
            const int lg = 32 - __clz(na - 1), G = 32 >> lg, g = lane >> (5 - lg), m = lane & (G - 1);
            const unsigned srcu = __fns(act, 0, g + 1);
            const bool has = srcu < 32u;
            const int src = has ? (int)srcu : lane;
            const int sa = __shfl_sync(0xffffffffu, a, src), saend = __shfl_sync(0xffffffffu, aend, src);
            int sbb = __shfl_sync(0xffffffffu, b, src);
            float su = __shfl_sync(0xffffffffu, u, src);
            const float sdmaj2f = __shfl_sync(0xffffffffu, R.dmaj2, src), sd8f = __shfl_sync(0xffffffffu, R.d8, src);
            const int sklo = __shfl_sync(0xffffffffu, klo, src);
            const bool sneg = __shfl_sync(0xffffffffu, (int)neg, src) != 0;
            const uint4 *sgtn = (const uint4 *)__shfl_sync(0xffffffffu, (unsigned long long)gtn, src);
            const int A = sa + 8 * m;
            const bool work = has && A <= saend;
            unsigned bad = 0u;
            if (work) {
                StripRay S;
                strip_ray_consts(S, sdmaj2f, sd8f);
                if (m > 0) {
                    const unsigned d2 = (unsigned)sdmaj2f, U = (unsigned)su + (unsigned)m * (unsigned)sd8f, steps = U / d2;
                    su = (float)(U - steps * d2);
                    sbb += sneg ? -(int)steps : (int)steps;
                }
                bad = strip_block(sgtn, tp, A, saend, m == 0 ? sklo : 0, sneg, S, sbb, su);
            }
            const unsigned badm = __ballot_sync(0xffffffffu, bad != 0u);
            // back to the owners: rank r among the active lanes = group r; the ray moves on G blocks
            const int r = __popc(act & lt);
            const int from = active ? r * G + G - 1 : lane;
            const int nb_ = __shfl_sync(0xffffffffu, sbb, from);
            const float nu_ = __shfl_sync(0xffffffffu, su, from);
            if (active) {
                const unsigned gm = (G == 32 ? 0xffffffffu : ((1u << G) - 1u)) << (r * G);
                const bool blocked = (badm & gm) != 0u;
                a += 8 * G;
                klo = 0;
                if (blocked || a > aend) {
                    out[idx] = blocked ? 0 : 1;
                    active = false;
                } else {
                    b = nb_;
                    u = nu_;
                }
            }
        }
    }
}

} // namespace trrt
