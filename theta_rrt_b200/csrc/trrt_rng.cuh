// trrt_rng.cuh -- numpy's legacy RandomState(seed).standard_normal(n) on the device, bit for bit, and the rand_conf
// samples drawn from such streams (rrt.py:53-68, samples.stream_from_normals).
//
// numpy's RandomState(int) seeds MT19937 with init_genrand; legacy_double takes two tempered words,
// ((a >> 5) * 2^26 + (b >> 6)) / 2^53; legacy_gauss is the polar method: x1 = 2d - 1, x2 = 2d - 1,
// r2 = x1*x1 + x2*x2 (unfused), rejected when r2 >= 1 or r2 == 0, f = sqrt(-2 log(r2) / r2), and a pair yields f*x2
// first and f*x1 second (standard_normal(n) with n odd keeps only f*x2 of the last pair).  Every candidate pair reads
// exactly 4 words whether it is accepted or not, so candidate j of a twist block reads words 4j..4j+3 and the 156
// candidates of a block are independent: the lanes of a warp evaluate 32 of them at once, and a ballot with a prefix
// popcount places the accepted ones.
//
// log(r2) is the host libm's in numpy.  tl_log_dd (trrt_libm.h) settles every log whose glibc rounding is forced;
// the pair of an undecided one gets x2 / x1 in its slots and an entry in the fixup list, and
// legacy_normals_fixup_kernel multiplies them by f once the host has evaluated those logs with its own libm.
#pragma once
#include "trrt_bike.cuh"

namespace trrt {

constexpr int MT_N = 624, MT_M = 397;
constexpr int MT_CAND = MT_N / 4; // candidate pairs per twist block
constexpr int RNG_WARPS = 4;      // warps (seeds in flight) per block of legacy_normals_kernel

struct LegacyNormalsDev {
    int64_t n;
    const uint32_t *seeds;   // [n]
    const int64_t *range;    // [n][2] = [begin, end) of seed i's normals in out
    double *out;
    int64_t *fix_pos;        // [fix_cap] slot of f*x2; ~slot when the pair's f*x1 slot does not exist
    double *fix_r2;          // [fix_cap]
    int64_t fix_cap;
    unsigned long long *fix_count;
    unsigned long long *next; // work counter (seeds handed out)
};

__device__ __forceinline__ uint32_t mt_temper(uint32_t y) {
    y ^= y >> 11;
    y ^= (y << 7) & 0x9d2c5680u;
    y ^= (y << 15) & 0xefc60000u;
    y ^= y >> 18;
    return y;
}

// One in-place MT19937 twist of mt[624] by one warp.  Word k reads mt[k], mt[k+1] (old) and mt[(k+397) % 624], which
// is old for k < 227, written by the first phase for k < 454 and by the second for the rest; k = 623 reads the new
// mt[0].  Within a phase every lane reads before any lane writes.
__device__ __forceinline__ void mt_twist_warp(uint32_t *mt, int lane) {
#pragma unroll 1
    for (int ph = 0; ph < 3; ph++) {
        const int lo = ph * (MT_N - MT_M), hi = ph == 2 ? MT_N : (ph + 1) * (MT_N - MT_M);
        for (int k0 = lo; k0 < hi; k0 += 32) {
            const int k = k0 + lane;
            uint32_t v = 0;
            if (k < hi) {
                const uint32_t y = (mt[k] & 0x80000000u) | (mt[k + 1 == MT_N ? 0 : k + 1] & 0x7fffffffu);
                const int km = k + MT_M < MT_N ? k + MT_M : k + MT_M - MT_N;
                v = mt[km] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
            }
            __syncwarp();
            if (k < hi) mt[k] = v;
            __syncwarp();
        }
    }
}

// Persistent warps: each takes the next seed from a.next and writes its normals.  Shared memory holds one MT state
// per warp.
__global__ void __launch_bounds__(RNG_WARPS * 32) legacy_normals_kernel(const LegacyNormalsDev a) {
    __shared__ __align__(16) uint32_t mt_all[RNG_WARPS][MT_N];
    const int lane = threadIdx.x & 31;
    uint32_t *mt = mt_all[threadIdx.x >> 5];
    const unsigned FULL = 0xffffffffu;
    for (;;) {
        unsigned long long q = 0;
        if (lane == 0) q = atomicAdd(a.next, 1ull);
        q = __shfl_sync(FULL, q, 0);
        if (q >= (unsigned long long)a.n) return;
        const int64_t begin = a.range[2 * q], cnt = a.range[2 * q + 1] - begin;
        if (cnt <= 0) continue;
        if (lane == 0) { // init_genrand: a sequential recurrence
            uint32_t s = a.seeds[q];
            mt[0] = s;
            for (int i = 1; i < MT_N; i++) {
                s = 1812433253u * (s ^ (s >> 30)) + (uint32_t)i;
                mt[i] = s;
            }
        }
        __syncwarp();
        int64_t placed = 0; // normals of this stream placed so far (2 per accepted pair)
        while (placed < cnt) {
            mt_twist_warp(mt, lane);
            for (int c0 = 0; c0 < MT_CAND && placed < cnt; c0 += 32) {
                const int c = c0 + lane;
                double x1 = 0.0, x2 = 0.0, r2 = 0.0;
                bool acc = false;
                if (c < MT_CAND) {
                    const uint4 w = reinterpret_cast<const uint4 *>(mt)[c];
                    const double d1 = __ddiv_rn(__dadd_rn((double)(mt_temper(w.x) >> 5) * 67108864.0, (double)(mt_temper(w.y) >> 6)),
                                                9007199254740992.0);
                    const double d2 = __ddiv_rn(__dadd_rn((double)(mt_temper(w.z) >> 5) * 67108864.0, (double)(mt_temper(w.w) >> 6)),
                                                9007199254740992.0);
                    x1 = __dadd_rn(__dmul_rn(2.0, d1), -1.0);
                    x2 = __dadd_rn(__dmul_rn(2.0, d2), -1.0);
                    r2 = __dadd_rn(__dmul_rn(x1, x1), __dmul_rn(x2, x2));
                    acc = r2 < 1.0 && r2 != 0.0;
                }
                const unsigned ball = __ballot_sync(FULL, acc);
                const int64_t p = placed + 2 * (int64_t)__popc(ball & ((1u << lane) - 1u)); // this pair's f*x2
                const bool mine = acc && p < cnt;
                bool undecided = false;
                if (mine) {
                    const int64_t o = begin + p;
                    const bool two = p + 1 < cnt;
                    TRRT_CHECK(p >= 0 && o + (two ? 1 : 0) < begin + cnt);
                    double hi, lo;
                    tl_log_dd(r2, &hi, &lo);
                    if (tl_log_decided(hi, lo)) {
                        const double f = __dsqrt_rn(__ddiv_rn(__dmul_rn(-2.0, hi), r2));
                        a.out[o] = __dmul_rn(f, x2);
                        if (two) a.out[o + 1] = __dmul_rn(f, x1);
                    } else {
                        a.out[o] = x2;
                        if (two) a.out[o + 1] = x1;
                        undecided = true;
                    }
                }
                // fixup entries: one atomic per warp and round
                const unsigned ub = __ballot_sync(FULL, undecided);
                if (ub) {
                    unsigned long long base = 0;
                    const int leader = __ffs(ub) - 1;
                    if (lane == leader) base = atomicAdd(a.fix_count, (unsigned long long)__popc(ub));
                    base = __shfl_sync(FULL, base, leader);
                    if (undecided) {
                        const unsigned long long k = base + __popc(ub & ((1u << lane) - 1u));
                        if (k < (unsigned long long)a.fix_cap) {
                            const int64_t o = begin + p;
                            TRRT_CHECK(k < (unsigned long long)a.fix_cap && o < begin + cnt);
                            a.fix_pos[k] = p + 1 < cnt ? o : ~o;
                            a.fix_r2[k] = r2;
                        }
                    }
                }
                placed += 2 * (int64_t)__popc(ball);
            }
        }
        __syncwarp(); // the next seed's init_genrand overwrites mt
    }
}

// The undecided pairs: f = sqrt(-2 log(r2) / r2) with the host's log, then f*x2 and f*x1 in place.
__global__ void legacy_normals_fixup_kernel(double *__restrict__ out, const int64_t *__restrict__ fix_pos, const double *__restrict__ fix_r2,
                                            const double *__restrict__ fix_log, int64_t n_fix) {
    for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < n_fix; k += (int64_t)gridDim.x * blockDim.x) {
        const int64_t p = fix_pos[k];
        const bool two = p >= 0;
        const int64_t o = two ? p : ~p;
        const double f = __dsqrt_rn(__ddiv_rn(__dmul_rn(-2.0, fix_log[k]), fix_r2[k]));
        out[o] = __dmul_rn(f, out[o]);
        if (two) out[o + 1] = __dmul_rn(f, out[o + 1]);
    }
}

// rrt.py:53-68 (samples.stream_from_normals) for one sample: the normals z[0..2] around the goal (gx, gy) with heading
// gth (already wrapped by standardangle): x = gx + (xystdv*H)*z0 clipped to [0, H-1] and truncated, theta wrapped.
__device__ __forceinline__ void rand_conf_sample(const double *z, double gx, double gy, double gth, double sx, double sy, double hm,
                                                 double wm, double anglestdv, int32_t &xi, int32_t &yi, double &th) {
    double x = gx + sx * z[0], y = gy + sy * z[1];
    x = x < 0.0 ? 0.0 : (x > hm ? hm : x);
    y = y < 0.0 ? 0.0 : (y > wm ? wm : y);
    xi = (int32_t)trunc_ll(x);
    yi = (int32_t)trunc_ll(y);
    th = standardangle(gth + anglestdv * z[2]);
}

// rand_conf streams of n queries, S samples each: query q reads normals[q*3S .. (q+1)*3S) and writes sample_xy
// (int32 or int16) [q][S][2] and sample_th [q][S], the layout trrt_rrt_batch takes.
template <typename XY>
__global__ void rand_conf_kernel(int H, int W, double xystdv, double anglestdv, int64_t n, int S, const double *__restrict__ goal,
                                 const double *__restrict__ normals, XY *__restrict__ sxy, double *__restrict__ sth) {
    const double sx = xystdv * (double)H, sy = xystdv * (double)W, hm = (double)(H - 1), wm = (double)(W - 1);
    const int64_t total = n * (int64_t)S;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t q = i / S;
        int32_t xi, yi;
        double th;
        rand_conf_sample(normals + 3 * i, goal[3 * q], goal[3 * q + 1], standardangle(goal[3 * q + 2]), sx, sy, hm, wm, anglestdv, xi, yi,
                         th);
        sxy[2 * i] = (XY)xi;
        sxy[2 * i + 1] = (XY)yi;
        sth[i] = th;
    }
}

} // namespace trrt
