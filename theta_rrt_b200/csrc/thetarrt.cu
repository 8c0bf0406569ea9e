// thetarrt.cu -- kernels and C ABI of libthetarrt.so (sm_100a).
//
// Kernels (one section each):
//   pack_grid_kernel      byte image -> bit-packed occupancy grid
//   los_batch_kernel      K4: search.lineofsight for independent segments, one thread per ray
//   tile_grid_kernel / los_tiled_kernel  K4b: the same test, 8 pixels per step over 8x16-pixel strips, per-lane refill (trrt_los.cuh)
//   nearest_tile_kernel   K1: fp64 argmin over SoA tree; query sets in registers, node slices per warp
//                             (the last CTA of a query group folds the per-column partials, lowest-index ties)
//   rrt_kernel_spec<G>    K2: fused rrt.rrt loop, speculative window of G iterations, persistent (trrt_rrt.cuh)
//   rrt_kernel_coop<G>        same loop, G lanes cooperating on one iteration at a time
//   steer / drive / arc batch kernels: single steps of K2 for the drop-in helpers and step-level parity tests
//   arc_pixels_kernel         pixel lists of search.getArc / getCircle / bresenham in the reference's list order
//   clearance / anglediff batch kernels: rrt.bike_clear, rrt.front_of_bike_clear, rrt.anglediff
//   findnearest_kernel    rrt.findnearest over the edge log
//   mission_*_kernel      main.py missions: segment chain around trrt_rrt_batch, findnearest restarts (trrt_mission.cuh)
//   theta_kernel<G>       K3: A* / lazy Theta*, G lanes per query, G-ary heap
//   legacy_normals_kernel / legacy_normals_fixup_kernel  numpy RandomState(seed).standard_normal streams (trrt_rng.cuh)
//   rand_conf_kernel<XY>  rrt.rand_conf samples from such streams
//
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -fmad=false -lineinfo
// (see theta_rrt_b200/build.py).  No tensor cores: nothing here is a dense
// contraction; the hot loops are fp64 compare/select and bit tests.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <string.h>

#include <algorithm>
#include <thread>
#include <vector>

#include "../../include/thetarrt.h"
#include "trrt_bike.cuh"
#include "trrt_device.cuh"
#include "trrt_los.cuh"
#include "trrt_mission.cuh"
#include "trrt_rng.cuh"
#include "trrt_rrt.cuh"

using namespace trrt;

static thread_local char g_last_cuda_error[256] = "";

static int cuda_fail(cudaError_t e) {
    if (e == cudaSuccess) return TRRT_OK;
    strncpy(g_last_cuda_error, cudaGetErrorString(e), sizeof(g_last_cuda_error) - 1);
    return (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver) ? TRRT_ERR_NO_DEVICE : TRRT_ERR_CUDA;
}
#define CUDA_TRY(x)                                  \
    do {                                             \
        cudaError_t e__ = (x);                       \
        if (e__ != cudaSuccess) return cuda_fail(e__); \
    } while (0)

static int check_map(int n_maps, int H, int W) {
    if (n_maps < 1 || H < 1 || W < 1) return TRRT_ERR_INVALID_ARGUMENT;
    if (H != W) return TRRT_ERR_NONSQUARE_MAP;
    if (H > 32768) return TRRT_ERR_MAP_TOO_LARGE;
    return TRRT_OK;
}

static int sm_count() {
    static int n = 0;
    if (n == 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess) return 148;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    }
    return n;
}

// ===========================================================================
// grid packing
// ===========================================================================
__global__ void pack_grid_kernel(const uint8_t *__restrict__ free_, int n_maps, int H, int W, int wpr, uint32_t *__restrict__ bits) {
    size_t total = (size_t)n_maps * H * wpr;
    for (size_t w = blockIdx.x * (size_t)blockDim.x + threadIdx.x; w < total; w += (size_t)gridDim.x * blockDim.x) {
        size_t row = w / wpr; // map * H + y
        int x0 = (int)(w % wpr) * 32;
        const uint8_t *src = free_ + row * (size_t)W;
        uint32_t v = 0;
        int lim = W - x0 < 32 ? W - x0 : 32;
        for (int b = 0; b < lim; b++) v |= (src[x0 + b] ? 1u : 0u) << b;
        bits[w] = v;
    }
}

// ===========================================================================
// K4 los_batch: one thread per segment, literal running-error Bresenham with
// four pixel probes in flight (the grid words come from L1/L2; the 8 MiB
// 8192^2 grid is L2 resident).
// ===========================================================================
__global__ void __launch_bounds__(256) los_batch_kernel(const uint32_t *__restrict__ bits, int H, int W, int wpr, const int32_t *__restrict__ map_id,
                                                        const int4 *__restrict__ seg, int64_t n, uint8_t *__restrict__ out) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    int4 s = __ldg(seg + i);
    int x0 = s.x, y0 = s.y, x1 = s.z, y1 = s.w;
    const uint32_t *g = bits + (map_id ? (size_t)__ldg(map_id + i) * H * wpr : 0);
    bool ok = x0 >= 0 && y0 >= 0 && x1 >= 0 && y1 >= 0 && x0 < H && x1 < H && y0 < W && y1 < W; // search.py:17-24
    if (ok) {
        int adx = abs(x1 - x0), ady = abs(y1 - y0);
        bool low = ady < adx; // search.py:47
        if (low ? (x0 > x1) : (y0 > y1)) { int t = x0; x0 = x1; x1 = t; t = y0; y0 = y1; y1 = t; }
        int dmaj = low ? adx : ady, dmin = low ? ady : adx;
        int step = low ? ((y1 < y0) ? -1 : 1) : ((x1 < x0) ? -1 : 1);
        int D = 2 * dmin - dmaj; // search.py:66 / :85
        int a = low ? x0 : y0, b = low ? y0 : x0, aend = a + dmaj;
        // word address pieces: low -> (x=a, y=b), high -> (x=b, y=a)
        while (a + 3 <= aend) {
            uint32_t acc = 0xffffffffu;
#pragma unroll
            for (int u = 0; u < 4; u++) {
                int px = low ? a : b, py = low ? b : a;
                uint32_t wv = __ldg(g + (size_t)py * wpr + (px >> 5));
                acc &= (wv >> (px & 31)) | 0xfffffffeu;
                if (D > 0) { b += step; D -= 2 * dmaj; }
                D += 2 * dmin;
                a++;
            }
            if (acc != 0xffffffffu) { ok = false; break; }
        }
        if (ok) {
            for (; a <= aend; a++) {
                int px = low ? a : b, py = low ? b : a;
                uint32_t wv = __ldg(g + (size_t)py * wpr + (px >> 5));
                if (!((wv >> (px & 31)) & 1u)) { ok = false; break; }
                if (D > 0) { b += step; D -= 2 * dmaj; }
                D += 2 * dmin;
            }
        }
    }
    out[i] = ok ? 1 : 0;
}

// ===========================================================================
// K1 nearest_batch
//   A CTA has 8 warps.  A warp owns one query set (TQ queries in registers) and one node slice; its lanes
//   stride the slice with 16-byte SoA loads (512 B per warp per array and load), four loads of x and four of y
//   in flight per lane.  With >= 8 query sets the warps of a CTA hold different sets and stream the same slice
//   (reuse through L1); with fewer sets the spare warps split the CTA's slice, so that a single query still puts
//   every warp of the GPU on the HBM stream.  Per-warp shuffle min-reduction ordered by (d2, index); partials go
//   to the workspace and the CTA that finishes last folds them (one warp per query).
//   d2 = rn(rn(dx*dx) + rn(dy*dy)), dx = qx - x  (search.py:15 before the sqrt).
// ===========================================================================
#define NN_WARPS 8
template <int TQ>
__device__ __forceinline__ void nn_fold(const double (&qx)[TQ], const double (&qy)[TQ], double (&bd)[TQ], int (&bi)[TQ], double2 xv, double2 yv,
                                        int i0) {
#pragma unroll
    for (int t = 0; t < TQ; t++) {
        double dx = qx[t] - xv.x, dy = qy[t] - yv.x;
        double d = dx * dx + dy * dy;
        if (d < bd[t]) { bd[t] = d; bi[t] = i0; }
        dx = qx[t] - xv.y; dy = qy[t] - yv.y;
        d = dx * dx + dy * dy;
        if (d < bd[t]) { bd[t] = d; bi[t] = i0 + 1; }
    }
}

template <int TQ>
__global__ void __launch_bounds__(NN_WARPS * 32) nearest_tile_kernel(const double *__restrict__ x, const double *__restrict__ y, int64_t n_nodes,
                                                                     const int32_t *__restrict__ qxy, int64_t n_q, int64_t slice_len, int spc_log2,
                                                                     double *part_d, int32_t *part_i, unsigned *done, int32_t *__restrict__ idx_out,
                                                                     double *__restrict__ d2_out) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int spc = 1 << spc_log2, wps = NN_WARPS >> spc_log2; // query sets per CTA, warps per set
    const int set_in_cta = warp & (spc - 1), sub = warp >> spc_log2;
    const int64_t q0 = ((int64_t)blockIdx.x * spc + set_in_cta) * TQ;
    const bool active = q0 < n_q;
    const int64_t slice = (int64_t)blockIdx.y * wps + sub;
    const int64_t lo = slice * slice_len;
    int64_t hi = lo + slice_len;
    if (hi > n_nodes) hi = n_nodes;
    double qx[TQ], qy[TQ], bd[TQ];
    int bi[TQ];
#pragma unroll
    for (int t = 0; t < TQ; t++) {
        int64_t q = q0 + t < n_q ? q0 + t : n_q - 1;
        qx[t] = (double)__ldg(qxy + 2 * q);
        qy[t] = (double)__ldg(qxy + 2 * q + 1);
        bd[t] = INFINITY;
        bi[t] = 0x7fffffff;
    }
    // slice_len is a multiple of 256 and x, y are 16-byte aligned (checked by the launcher): double2 loads
    const double2 *x2 = reinterpret_cast<const double2 *>(x);
    const double2 *y2 = reinterpret_cast<const double2 *>(y);
    int64_t p = (lo >> 1) + lane;
    const int64_t pend = (active && hi > lo) ? (hi >> 1) : 0; // pair index
    for (; p + 96 < pend; p += 128) {
        const double2 xa = __ldg(x2 + p), xb = __ldg(x2 + p + 32), xc = __ldg(x2 + p + 64), xd = __ldg(x2 + p + 96);
        const double2 ya = __ldg(y2 + p), yb = __ldg(y2 + p + 32), yc = __ldg(y2 + p + 64), yd = __ldg(y2 + p + 96);
        const int i0 = (int)(p << 1);
        nn_fold<TQ>(qx, qy, bd, bi, xa, ya, i0);
        nn_fold<TQ>(qx, qy, bd, bi, xb, yb, i0 + 64);
        nn_fold<TQ>(qx, qy, bd, bi, xc, yc, i0 + 128);
        nn_fold<TQ>(qx, qy, bd, bi, xd, yd, i0 + 192);
    }
    for (; p < pend; p += 32) nn_fold<TQ>(qx, qy, bd, bi, __ldg(x2 + p), __ldg(y2 + p), (int)(p << 1));
    if (active && (hi & 1) && lane == 0 && hi == n_nodes && hi > lo) { // odd tail node of the last slice
        int i0 = (int)(hi - 1);
        double xs = __ldg(x + i0), ys = __ldg(y + i0);
#pragma unroll
        for (int t = 0; t < TQ; t++) {
            double dx = qx[t] - xs, dy = qy[t] - ys;
            double d = dx * dx + dy * dy;
            if (d < bd[t] || (d == bd[t] && i0 < bi[t])) { bd[t] = d; bi[t] = i0; }
        }
    }
    __shared__ double sd[NN_WARPS][TQ];
    __shared__ int si[NN_WARPS][TQ];
#pragma unroll
    for (int t = 0; t < TQ; t++) {
        double d = bd[t];
        int i = bi[t];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            double od = __shfl_xor_sync(0xffffffffu, d, off);
            int oi = __shfl_xor_sync(0xffffffffu, i, off);
            if (od < d || (od == d && oi < i)) { d = od; i = oi; }
        }
        if (lane == 0) { sd[warp][t] = d; si[warp][t] = i; }
    }
    __syncthreads();
    // the warps of one query set fold their sub-slices: one partial per (CTA column, query)
    if (sub == 0 && active && lane < TQ && q0 + lane < n_q) {
        double d = sd[warp][lane];
        int i = si[warp][lane];
        for (int w = 1; w < wps; w++) {
            double od = sd[set_in_cta + (w << spc_log2)][lane];
            int oi = si[set_in_cta + (w << spc_log2)][lane];
            if (od < d || (od == d && oi < i)) { d = od; i = oi; }
        }
        part_d[(int64_t)blockIdx.y * n_q + q0 + lane] = d;
        part_i[(int64_t)blockIdx.y * n_q + q0 + lane] = i;
        __threadfence(); // the partial is visible before this CTA is counted
    }
    // The CTA that finishes last among those sharing this query group folds the per-column partials (no second launch:
    // a single-query scan is ~45 us, a launch plus a tiny kernel behind it ~10 us).  (d2, index) order makes the fold
    // order irrelevant.
    __shared__ bool last;
    __syncthreads();
    if (threadIdx.x == 0) last = atomicAdd(done + blockIdx.x, 1u) == gridDim.y - 1;
    __syncthreads();
    if (!last) return;
    __threadfence();
    const int n_slices = (int)gridDim.y;
    const int64_t qa = (int64_t)blockIdx.x * spc * TQ;
    for (int64_t q = qa + warp; q < qa + (int64_t)spc * TQ && q < n_q; q += NN_WARPS) {
        double bd = INFINITY;
        int bi = 0x7fffffff;
        for (int sidx = lane; sidx < n_slices; sidx += 32) {
            const double d = __ldcg(part_d + (int64_t)sidx * n_q + q);
            const int i = __ldcg(part_i + (int64_t)sidx * n_q + q);
            if (d < bd || (d == bd && i < bi)) { bd = d; bi = i; }
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            const double od = __shfl_xor_sync(0xffffffffu, bd, off);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, off);
            if (od < bd || (od == bd && oi < bi)) { bd = od; bi = oi; }
        }
        if (lane == 0) {
            idx_out[q] = (bi == 0x7fffffff) ? -1 : bi;
            if (d2_out) d2_out[q] = bd;
        }
    }
}

// ===========================================================================
// Single-step entry points: rrt.steer / rrt.drive / the rrt.py:173-174 edge
// test for batches of independent inputs (one thread each).  They run exactly
// the device functions the fused kernel uses.
// ===========================================================================
__global__ void steer_batch_kernel(BikeParams P, int64_t n, const double *__restrict__ in, double *__restrict__ out, uint8_t *__restrict__ straight) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    Steer s;
    steer(P, in[6 * i], in[6 * i + 1], in[6 * i + 2], in[6 * i + 3], in[6 * i + 4], in[6 * i + 5], s);
    double *o = out + 8 * i;
    o[0] = s.x; o[1] = s.y; o[2] = s.theta; o[3] = s.steer; o[4] = s.iccx; o[5] = s.iccy; o[6] = s.rad; o[7] = s.dist;
    straight[i] = s.straight ? 1 : 0;
}
__global__ void drive_batch_kernel(BikeParams P, int64_t n, const double *__restrict__ in, double *__restrict__ out) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double *v = in + 8 * i;
    double fx, fy, fa;
    drive(P, v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7], fx, fy, fa);
    out[3 * i] = fx; out[3 * i + 1] = fy; out[3 * i + 2] = fa;
}
template <int G>
__global__ void arc_batch_kernel(const uint32_t *__restrict__ bits, int H, int W, int wpr, const int32_t *__restrict__ map_id, int64_t n,
                                 const double *__restrict__ in, uint8_t *__restrict__ blocked) {
    const Group<G> g;
    int64_t i = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / G;
    if (i >= n) return;
    Grid m;
    m.W = W; m.H = H; m.wpr = wpr;
    m.bits = bits + (map_id ? (size_t)map_id[i] * H * wpr : 0);
    const double *v = in + 9 * i;
    bool b;
    if (v[8] != 0.0) b = !los_group<G>(g, m, trunc_ll(v[0]), trunc_ll(v[1]), trunc_ll(v[2]), trunc_ll(v[3]));
    else b = arc_blocked<G>(g, m, v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7], nullptr, nullptr);
    if (g.gl == 0) blocked[i] = b ? 1 : 0;
}

// ===========================================================================
// Pixel lists of the raster helpers, in the reference's own list order (duplicates included), one warp per item:
//   mode 0  search.getArc(begin, land, u) for a curved edge        (search.py:144-182)
//   mode 1  search.bresenham(begin, land) / getArc of a straight u (search.py:43-94, :145-146)
//   mode 2  search.getCircle(center = icc, r = rad)                (search.py:96-142)
// getCircle's loop emits, for y = 0 .. t_max, getCirclePoints(xc, yc, x_y, y): the offsets (v1, v2) with v1, v2 drawn in
// order from [-p, p, -q, q] and |v1| != |v2|, i.e. (-p,-q) (-p,q) (p,-q) (p,q) (-q,-p) (-q,p) (q,-p) (q,p) -- for q = 0
// that list holds every pixel twice, and so does the reference's.  Pixels outside the image are dropped (search.py:103),
// then getArc keeps those inside the arc's angular span (arc_keeps_pixel).  Lane l of the warp owns row base + l; a warp
// prefix sum of the rows' pixel counts gives every pixel its position in the list.
// d_in [n][9] = begin x, y, land x, y, u.steer, icc x, icc y, rad, mode.  d_count[i] = length of the full list even when
// it exceeds cap (the caller then calls again with a larger cap); d_pixels [n][cap][2].
// ===========================================================================
__global__ void __launch_bounds__(128) arc_pixels_kernel(int H, int W, int64_t n, const double *__restrict__ in, int cap,
                                                         int32_t *__restrict__ pixels, int32_t *__restrict__ count) {
    const int lane = threadIdx.x & 31;
    const int64_t item = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (item >= n) return;
    const double *v = in + 9 * item;
    int32_t *out = pixels + item * (int64_t)cap * 2;
    const int mode = (int)v[8];
    long long total = 0;
    auto emit = [&](int my_cnt, const int *px, const int *py) { // my_cnt pixels of this lane, lanes in order
        int inc = my_cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
        const long long base = total + inc - my_cnt;
        for (int k = 0; k < my_cnt; k++)
            if (base + k < cap) { out[2 * (base + k)] = px[k]; out[2 * (base + k) + 1] = py[k]; }
        total += __shfl_sync(0xffffffffu, inc, 31);
    };
    if (mode == 1) { // search.py:43-94
        long long x0 = trunc_ll(v[0]), y0 = trunc_ll(v[1]), x1 = trunc_ll(v[2]), y1 = trunc_ll(v[3]);
        const long long adx = llabs(x1 - x0), ady = llabs(y1 - y0);
        const bool low = ady < adx;
        if (low ? (x0 > x1) : (y0 > y1)) { long long t = x0; x0 = x1; x1 = t; t = y0; y0 = y1; y1 = t; }
        const long long dmaj = low ? adx : ady, dmin = low ? ady : adx;
        const long long step = low ? ((y1 < y0) ? -1 : 1) : ((x1 < x0) ? -1 : 1);
        for (long long base = 0; base <= dmaj; base += 32) {
            const long long i = base + lane;
            int px[1], py[1], c = 0;
            if (i <= dmaj) {
                const long long sm = dmaj ? (2 * dmin * i + dmaj - 1) / (2 * dmaj) : 0; // DESIGN.md 8.1
                px[0] = (int)(low ? x0 + i : x0 + step * sm);
                py[0] = (int)(low ? y0 + step * sm : y0 + i);
                c = 1;
            }
            emit(c, px, py);
        }
    } else {
        Grid m;
        m.W = W; m.H = H; m.wpr = 0; m.bits = nullptr;
        const double bx = v[0], by = v[1], lx = v[2], ly = v[3];
        const long long xc = trunc_ll(v[5]), yc = trunc_ll(v[6]), r = trunc_ll(v[7]);
        ArcTest A;
        A.iccx = v[5]; A.iccy = v[6]; A.usteer = v[4]; A.ready = false;
        const long long tmax = circle_tmax(r);
        for (long long base = 0; base <= tmax; base += 32) {
            const long long t = base + lane;
            int px[8], py[8], c = 0;
            if (t <= tmax) {
                const long long x = (t == 0) ? r : circle_x(r, t);
                const long long o1[8] = {-x, -x, x, x, -t, -t, t, t}, o2[8] = {-t, t, -t, t, -x, x, -x, x};
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    const long long qx = xc + o1[k], qy = yc + o2[k];
                    if (!m.inb(qx, qy)) continue;
                    if (mode == 0 && !arc_keeps_pixel(A, bx, by, lx, ly, qx, qy)) continue;
                    px[c] = (int)qx; py[c] = (int)qy; c++;
                }
            }
            emit(c, px, py);
        }
        // diagonal-gap pixels (search.py:124-138)
        const long long rnd = py_round((double)r * 0.5 * sqrt(2.0));
        bool drawmore = true;
        {
            const int nx[4] = {1, -1, 0, 0}, ny[4] = {0, 0, 1, -1};
#pragma unroll
            for (int i = 0; i < 4; i++) {
                const long long a = rnd + nx[i], b = rnd + ny[i];
                if (m.inb(xc + a, yc + b) && circle_member(r, a, b)) drawmore = false;
            }
        }
        if (drawmore) {
            int px[1], py[1], c = 0;
            if (lane < 4) { // (+,+) (-,-) (+,-) (-,+)
                const long long qx = xc + ((lane == 0 || lane == 2) ? rnd : -rnd), qy = yc + ((lane == 0 || lane == 3) ? rnd : -rnd);
                if (m.inb(qx, qy) && (mode != 0 || arc_keeps_pixel(A, bx, by, lx, ly, qx, qy))) { px[0] = (int)qx; py[0] = (int)qy; c = 1; }
            }
            emit(c, px, py);
        }
    }
    if (lane == 0) count[item] = (int32_t)(total > 0x7fffffff ? 0x7fffffff : total);
}

// rrt.bike_clear / rrt.front_of_bike_clear (rrt.py:208-222) and rrt.anglediff (rrt.py:108-115) for batches:
//   in [n][3] = x, y, theta  ->  clear [n][2] = bike_clear, front_of_bike_clear
//   ang [n][2] = a1, a2      ->  diff [n]
__global__ void clearance_batch_kernel(const uint32_t *__restrict__ bits, int H, int W, int wpr, const int32_t *__restrict__ map_id, BikeParams P,
                                       int64_t n, const double *__restrict__ in, uint8_t *__restrict__ clear) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    Grid m;
    m.W = W; m.H = H; m.wpr = wpr;
    m.bits = bits + (map_id ? (size_t)map_id[i] * H * wpr : 0);
    const double x = in[3 * i], y = in[3 * i + 1], th = in[3 * i + 2];
    const Rot R = rot_make(th);
    double bx, by;
    rot_apply(R, P.bikelength, 0.0, bx, by);
    clear[2 * i] = los_lane(m, trunc_ll(x), trunc_ll(y), trunc_ll(bx + x), trunc_ll(by + y)) ? 1 : 0;
    rot_apply(R, P.bikelength * P.frontclearance, 0.0, bx, by);
    clear[2 * i + 1] = los_lane(m, trunc_ll(x), trunc_ll(y), trunc_ll(bx + x), trunc_ll(by + y)) ? 1 : 0;
}
__global__ void anglediff_batch_kernel(int64_t n, const double *__restrict__ in, double *__restrict__ out) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) out[i] = anglediff(in[2 * i], in[2 * i + 1]);
}

// ===========================================================================
// rrt.findnearest (rrt.py:117-128): one block per query over the edge log
// (findnearest_block, trrt_mission.cuh).
// ===========================================================================
__global__ void __launch_bounds__(FN_THREADS) findnearest_kernel(BikeParams P, int64_t nq, int K, const double *__restrict__ nx, const double *__restrict__ ny,
                                                                 const double *__restrict__ nth, const int32_t *__restrict__ it_near,
                                                                 const int32_t *__restrict__ it_new, const double *__restrict__ goal, int32_t *best,
                                                                 double *best_dist) {
    int64_t q = blockIdx.x;
    int b;
    double d;
    findnearest_block(P, K, nx + q * K, ny + q * K, nth + q * K, it_near + q * (int64_t)(K - 1), it_new + q * (int64_t)(K - 1), goal[3 * q],
                      goal[3 * q + 1], goal[3 * q + 2], b, d);
    if (threadIdx.x == 0) { best[q] = b; best_dist[q] = d; }
}

// ===========================================================================
// K3 theta_batch: A* / lazy Theta* (search.py:221-307), G >= 8 lanes per query.
// Per-slot state in the workspace:
//   cells[H*W]  {g fp64, parent int32, stamp uint32}; stamp = epoch<<2 | closed<<1 | open,
//               an entry belongs to the running query only when its epoch matches
//   heap[cap]   {f fp64, cell uint32}; cell index = x*W + y, so (f, cell) order is the
//               reference's tuple order (f, (x, y))
// Lane j < 8 owns neighbour j of the expanded node (order of search.py:187).
// ===========================================================================
struct __align__(16) Cell { double g; int parent; unsigned stamp; };
struct __align__(16) HeapEnt { double f; unsigned c; unsigned pad; };

struct ThetaDev {
    const uint32_t *bits;
    int H, W, wpr;
    const int32_t *map_id;
    int thetastar;
    int64_t nq;
    const int32_t *sg;
    int32_t *path;
    int path_cap;
    int32_t *path_len;
    double *cost;
    int32_t *expanded, *status;
    uint8_t *los_log;
    int los_cap;
    int32_t *n_los, *pushes;
    int n_slots, heap_cap;
    Cell *cells;
    HeapEnt *heap;
    unsigned long long *next_query; // dynamic query counter
    const int32_t *order;           // optional dispatch order
};

__device__ __forceinline__ bool hless(double f1, unsigned c1, double f2, unsigned c2) { return f1 < f2 || (f1 == f2 && c1 < c2); }

// The open list is a G-ary heap (G = lanes of the group): node i has children G*i+1 .. G*i+G.  A pop descends
// log_G(size) levels (3 for the 2 800 entries of the map2 query with G = 32) and at each level the G children are
// read with one coalesced load and reduced with shuffles, instead of the ~12 dependent compare-and-swap rounds one
// lane would spend in a binary heap.  Pushes climb at most the same levels (leader only).  The whole heap lives in the
// query slot's part of the global workspace, one 16-byte entry per position; its top levels stay resident in L1.
// Keeping the top three levels (1 + G + G*G entries) in shared memory instead was measured slower on B200: 292 ms
// vs 241 ms for 2048 map2 queries.  Any correct min-heap on the total order (f, cell) pops in the reference's
// PriorityQueue order (search.py:231,249).
template <int G>
struct Heap {
    HeapEnt *gh; // indexed by heap position
    __device__ __forceinline__ void get(int i, double &f, unsigned &c) const {
        HeapEnt e = gh[i]; f = e.f; c = e.c;
    }
    __device__ __forceinline__ void put(int i, double f, unsigned c) const {
        HeapEnt e; e.f = f; e.c = c; e.pad = 0; gh[i] = e;
    }
};

template <int G>
__device__ __forceinline__ bool heap_push(const Heap<G> &h, int &size, int cap, double f, unsigned c) {
    if (size >= cap) return false;
    int i = size++;
    TRRT_CHECK(i >= 0 && i < cap);
    while (i > 0) {
        const int p = (i - 1) / G;
        double pf;
        unsigned pc;
        h.get(p, pf, pc);
        if (!hless(f, c, pf, pc)) break;
        h.put(i, pf, pc);
        i = p;
    }
    h.put(i, f, c);
    return true;
}
// cooperative pop: every lane of the group calls it with the same arguments and receives the same result.
// f >= 0 always (sums of distances), so the IEEE bit pattern of f orders like f and the group minimum of
// (f, cell) is three 32-bit warp reductions (REDUX) -- high word, low word, cell -- each over the lanes still tied.
template <int G>
__device__ __forceinline__ void heap_pop(const Group<G> &g, const Heap<G> &h, int &size, double &top_f, unsigned &top_c) {
    h.get(0, top_f, top_c);
    double lf;
    unsigned lc;
    h.get(--size, lf, lc);
    const int base = (threadIdx.x & 31) & ~(G - 1);
    int i = 0;
    for (;;) {
        const int fc = G * i + 1;
        if (fc >= size) break;
        double bf = INFINITY;
        unsigned bc = 0xffffffffu;
        if (fc + g.gl < size) h.get(fc + g.gl, bf, bc);
        const unsigned long long kb = (unsigned long long)__double_as_longlong(bf);
        const unsigned hi = (unsigned)(kb >> 32), lo = (unsigned)kb;
        const unsigned mh = __reduce_min_sync(g.mask, hi);
        bool cand = hi == mh;
        const unsigned ml = __reduce_min_sync(g.mask, cand ? lo : 0xffffffffu);
        cand = cand && lo == ml;
        const unsigned mc = __reduce_min_sync(g.mask, cand ? bc : 0xffffffffu);
        cand = cand && bc == mc;
        const int bl = __ffs(__ballot_sync(g.mask, cand) & g.mask) - 1 - base; // equal keys are interchangeable
        const double mf = __longlong_as_double((long long)(((unsigned long long)mh << 32) | ml));
        if (!hless(mf, mc, lf, lc)) break;
        if (g.gl == 0) h.put(i, mf, mc);
        i = fc + bl;
    }
    g.sync(); // children were read by all lanes before the leader overwrites a slot on the path
    if (size > 0 && g.gl == 0) h.put(i, lf, lc);
    g.sync();
}

// Cells are named by pk = (x << 16) | y: the same order as the reference's (x, y) tuples, no division to get the
// coordinates back, and x*W + y is one multiply-add when the per-cell record is needed.
__device__ __forceinline__ unsigned pk_of(int x, int y) { return ((unsigned)x << 16) | (unsigned)y; }
__device__ __forceinline__ int pk_x(unsigned pk) { return (int)(pk >> 16); }
__device__ __forceinline__ int pk_y(unsigned pk) { return (int)(pk & 0xffffu); }

template <int G>
__global__ void __launch_bounds__(128) theta_kernel(const ThetaDev a) {
    static_assert(G >= 8, "one lane per neighbour");
    const Group<G> g;
    const int slot = (int)((blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / G);
    if (slot >= a.n_slots) return;
    const bool lead = g.gl == 0;
    const int W = a.W, H = a.H;
    Cell *cells = a.cells + (size_t)slot * H * W;
    Heap<G> heap;
    heap.gh = a.heap + (size_t)slot * a.heap_cap;
    const int base_lane = (threadIdx.x & 31) & ~(G - 1);
    // neighbour j = node - delta_j, delta in itertools.product([-1,0,1], repeat=2) minus (0,0)  (search.py:187-189)
    const int j = g.gl & 7;
    const int ndx = (j < 3) ? 1 : (j < 5 ? 0 : -1);
    const int ndy = (j == 0 || j == 3 || j == 5) ? 1 : ((j == 1 || j == 6) ? 0 : -1);
    const double ndist = (ndx != 0 && ndy != 0) ? sqrt(2.0) : 1.0; // L2norm of a unit step
    unsigned epoch = 0;
    for (;;) {
        unsigned long long qq = 0;
        if (lead) qq = atomicAdd(a.next_query, 1ull);
        qq = g.bcast(qq, 0);
        if (qq >= (unsigned long long)a.nq) break;
        const int64_t q = a.order ? (int64_t)a.order[qq] : (int64_t)qq;
        epoch++;
        Grid m;
        m.W = W; m.H = H; m.wpr = a.wpr;
        m.bits = a.bits + (a.map_id ? (size_t)a.map_id[q] * H * a.wpr : 0);
        const int sx = a.sg[4 * q], sy = a.sg[4 * q + 1], gx = a.sg[4 * q + 2], gy = a.sg[4 * q + 3];
        uint8_t *los_log = a.los_log ? a.los_log + q * (int64_t)a.los_cap : nullptr;
        int status = TRRT_OK_NOT_FOUND, nlos = 0, npush = 0, nclosed = 0, hsize = 0;
        bool overflow = false;
        if (!m.inb(sx, sy) || !m.inb(gx, gy)) status = TRRT_ERR_ENDPOINT_INVALID;                  // search.py:222
        else if (!m.free_nb(sx, sy) || !m.free_nb(gx, gy)) status = TRRT_ERR_ENDPOINT_BLOCKED;    // search.py:225
        const unsigned goal_c = pk_of(gx, gy);
        if (status == TRRT_OK_NOT_FOUND) {
            const unsigned sc = pk_of(sx, sy);
            // seed: expand the start node (search.py:237-244)
            double pf = 0;
            unsigned pc = 0;
            bool has = false;
            if (g.gl < 8) {
                int x = sx + ndx, y = sy + ndy;
                if (m.freespace(x, y)) {
                    Cell v; v.g = ndist; v.parent = (int)sc; v.stamp = (epoch << 2) | 1u;
                    cells[x * W + y] = v;
                    double hx = (double)(gx - x), hy = (double)(gy - y);
                    pf = ndist + sqrt(hx * hx + hy * hy);
                    pc = pk_of(x, y); has = true;
                }
            }
            if (lead) { Cell v; v.g = 0.0; v.parent = -1; v.stamp = (epoch << 2) | 2u; cells[sx * W + sy] = v; }
            nclosed = 1;
            for (int t = 0; t < 8; t++) {
                bool h1 = g.bcast(has, t); double f1 = g.bcast(pf, t); unsigned c1 = g.bcast(pc, t);
                if (h1) { if (lead && !heap_push<G>(heap, hsize, a.heap_cap, f1, c1)) overflow = true; npush++; }
            }
            hsize = g.bcast(hsize, 0);
            overflow = g.bcast(overflow, 0);
            g.sync();
            // main loop (search.py:247-304)
            while (hsize > 0 && !overflow) {
                double top_f;
                unsigned cur;
                heap_pop<G>(g, heap, hsize, top_f, cur); // hsize stays uniform: every lane decrements its copy
                const int cx = pk_x(cur), cy = pk_y(cur);
                const int cur_i = cx * W + cy;
                TRRT_CHECK(cx >= 0 && cx < H && cy >= 0 && cy < W && hsize >= 0 && hsize < a.heap_cap);
                Cell cc = cells[cur_i];
                // The records of the 8 neighbours are needed twice below (parent repair, relaxation) and nothing this group
                // writes in between touches them, so lane j asks for neighbour j's record NOW: the loads (L2 most of the
                // time: 1.4 MB of cells per search on map2) travel while the parent's line of sight is being walked.
                bool nfree = false;
                int nci = 0, nx_ = cx + ndx, ny_ = cy + ndy;
                Cell nbp;
                nbp.g = 0.0; nbp.parent = 0; nbp.stamp = 0u;
                if (g.gl < 8 && m.inb(nx_, ny_)) {
                    nci = nx_ * W + ny_;
                    TRRT_CHECK(nci >= 0 && nci < H * W);
                    nbp = cells[nci];
                    nfree = m.free_nb(nx_, ny_);
                }
                if (cc.stamp & 2u) continue; // already closed: stale heap copy (search.py:250-255); epoch matches by construction
                double gpar = 0.0;
                if (a.thetastar) { // search.py:258-263
                    const int px = pk_x((unsigned)cc.parent), py = pk_y((unsigned)cc.parent);
                    gpar = cells[px * W + py].g; // g of the parent (search.py:295), asked for before the ray walk
                    bool los = los_group<G>(g, m, cx, cy, px, py);
                    if (los_log && lead && nlos < a.los_cap) los_log[nlos] = los ? 1 : 0;
                    nlos++;
                    if (!los) {
                        double v = INFINITY;
                        int vi = 0x7fffffff;
                        unsigned vc = 0;
                        if (nfree && (nbp.stamp >> 2) == epoch && (nbp.stamp & 2u)) { v = nbp.g + ndist; vi = j; vc = pk_of(nx_, ny_); }
                        double bv = v;
                        int bj = vi;
                        g.min_di(bv, bj);
                        if (bj == 0x7fffffff) { status = TRRT_ERR_REF_RAISES_ARGMIN_EMPTY; break; }
                        unsigned bc = g.bcast(vc, bj);
                        cc.parent = (int)bc;
                        cc.g = bv;
                        gpar = g.bcast(nbp.g, bj); // the new parent is that closed neighbour
                    }
                }
                cc.stamp = (epoch << 2) | 2u; // openSet.remove, closedSet.add (search.py:265-266)
                g.sync(); // every lane has read cells[cur] (lanes are not in lockstep) before the leader rewrites it
                if (lead) cells[cur_i] = cc;
                nclosed++;
                if (cur == goal_c) { status = TRRT_OK_FOUND; break; }
                // neighbours (search.py:274-304), one lane each
                const unsigned pcell = (unsigned)cc.parent;
                const int ppx = pk_x(pcell), ppy = pk_y(pcell);
                int np_ = 0;
                double f1 = 0, f2 = 0;
                unsigned nbc = 0;
                {
                    const int x = nx_, y = ny_;
                    if (nfree) {
                        const int ci = nci;
                        Cell nb = nbp;
                        bool mine = (nb.stamp >> 2) == epoch;
                        bool closed = mine && (nb.stamp & 2u);
                        if (!closed) {
                            bool open = mine && (nb.stamp & 1u);
                            double hx = (double)(gx - x), hy = (double)(gy - y);
                            double hh = sqrt(hx * hx + hy * hy);
                            double gn = cc.g + ndist;
                            bool dirty = false;
                            if (!open) { nb.g = gn; nb.parent = (int)cur; nb.stamp = (epoch << 2) | 1u; f1 = gn + hh; np_ = 1; dirty = true; }
                            else if (gn < nb.g) { nb.g = gn; nb.parent = (int)cur; f1 = gn + hh; np_ = 1; dirty = true; }
                            if (a.thetastar) {
                                double ex = (double)(x - ppx), ey = (double)(y - ppy);
                                double g2 = gpar + sqrt(ex * ex + ey * ey);
                                if (g2 < nb.g) {
                                    nb.parent = (int)pcell; nb.g = g2; dirty = true;
                                    if (np_ == 0) { f1 = g2 + hh; np_ = 1; } else { f2 = g2 + hh; np_ = 2; }
                                }
                            }
                            if (dirty) cells[ci] = nb;
                            nbc = pk_of(x, y);
                        }
                    }
                }
                // pushes in neighbour order (search.py:279-304): only the lanes that have one
                unsigned todo = (__ballot_sync(g.mask, np_ > 0) & g.mask) >> base_lane;
                while (todo) {
                    const int t = __ffs(todo) - 1;
                    todo &= todo - 1;
                    const int cnt = g.bcast(np_, t);
                    const double fa = g.bcast(f1, t), fb = g.bcast(f2, t);
                    const unsigned c1 = g.bcast(nbc, t);
                    // The reference puts (fa, node) and then, when the grand-parent path is shorter, (fb, node) with
                    // fb <= fa (search.py:283-304).  The node is closed when its smallest entry is popped and every later
                    // pop of it is skipped (search.py:250-255), so the (fa, node) entry of such a pair can never act:
                    // only the smaller key is stored; `pushes` still counts what the reference puts.
                    if (lead && !heap_push<G>(heap, hsize, a.heap_cap, cnt == 2 ? fb : fa, c1)) overflow = true;
                    npush += cnt;
                }
                hsize = g.bcast(hsize, 0);
                overflow = g.bcast(overflow, 0);
                g.sync();
            }
            if (overflow) status = TRRT_ERR_CAPACITY;
        }
        g.sync();
        // reconstruct (search.py:196-204) + cost, by the leader; the global heap array is free now and serves as scratch
        if (lead) {
            int len = 0;
            double cost = 0.0;
            if (status == TRRT_OK_FOUND) {
                unsigned c = goal_c;
                unsigned *scratch = reinterpret_cast<unsigned *>(heap.gh);
                const long long scap = (long long)a.heap_cap * 4;
                for (;;) {
                    if (len < scap) scratch[len] = c;
                    len++;
                    int p = cells[pk_x(c) * W + pk_y(c)].parent;
                    if (p < 0) break;
                    c = (unsigned)p;
                }
                if (len > scap) status = TRRT_ERR_CAPACITY;
                else {
                    int32_t *path = a.path ? a.path + q * (int64_t)a.path_cap * 2 : nullptr;
                    int ppx = 0, ppy = 0;
                    for (int i = 0; i < len; i++) {
                        unsigned cidx = scratch[len - 1 - i];
                        int x = pk_x(cidx), y = pk_y(cidx);
                        if (path && i < a.path_cap) { path[2 * i] = x; path[2 * i + 1] = y; }
                        if (i > 0) { double ex = (double)(x - ppx), ey = (double)(y - ppy); cost += sqrt(ex * ex + ey * ey); }
                        ppx = x; ppy = y;
                    }
                }
            }
            a.path_len[q] = len;
            a.cost[q] = cost;
            a.expanded[q] = (status == TRRT_OK_FOUND) ? nclosed : 0;
            a.status[q] = status;
            if (a.n_los) a.n_los[q] = nlos;
            if (a.pushes) a.pushes[q] = npush;
        }
        g.sync();
    }
}

// Workspace of mission_batch: per-mission state, then the per-slot rows of one stage (trrt_rrt_batch inputs and
// outputs for up to n_missions slots), then trrt_rrt_batch's own workspace; every region starts 256-byte aligned.
struct MissionCarve {
    char *base;
    size_t p;
    template <typename T> T *take(size_t count) {
        p = (p + 255) & ~(size_t)255;
        T *r = base ? (T *)(base + p) : nullptr;
        p += count * sizeof(T);
        return r;
    }
};
static size_t mission_carve(MissionDev &d, void *work, int64_t n, int K) {
    MissionCarve c{(char *)work, 0};
    const size_t N = (size_t)n, Kn = (size_t)K, K1 = (size_t)(K - 1);
    d.off = c.take<int64_t>(N); d.restart = c.take<double>(3 * N); d.restarted = c.take<int32_t>(N);
    d.q_start = c.take<double>(3 * N); d.q_goal = c.take<double>(3 * N); d.q_map = c.take<int32_t>(N);
    d.q_sxy = c.take<int32_t>(2 * N * K1); d.q_sth = c.take<double>(N * K1);
    d.nx = c.take<double>(N * Kn); d.ny = c.take<double>(N * Kn); d.nth = c.take<double>(N * Kn); d.u = c.take<double>(5 * N * Kn);
    d.parent = c.take<int32_t>(N * Kn);
    d.q_n_nodes = c.take<int32_t>(N); d.q_sol = c.take<int32_t>(N); d.q_status = c.take<int32_t>(N); d.q_iters = c.take<int32_t>(N);
    d.it_near = c.take<int32_t>(N * K1); d.it_new = c.take<int32_t>(N * K1);
    c.take<char>(0); // start of the RRT workspace
    return c.p;
}

// ===========================================================================
// C ABI
// ===========================================================================
extern "C" {

int trrt_version(void) { return TRRT_VERSION; }

const char *trrt_error_string(int err) {
    switch (err) {
    case TRRT_OK: return "ok";
    case TRRT_ERR_INVALID_ARGUMENT: return "invalid argument";
    case TRRT_ERR_NONSQUARE_MAP: return "map must be square (reference bounds test, search.py:21)";
    case TRRT_ERR_MAP_TOO_LARGE: return "map side exceeds 32768";
    case TRRT_ERR_WORKSPACE_TOO_SMALL: return "workspace too small";
    case TRRT_ERR_CUDA: return "CUDA error (see trrt_last_cuda_error)";
    case TRRT_ERR_NO_DEVICE: return "no CUDA device";
    default: return "unknown error";
    }
}
const char *trrt_last_cuda_error(void) { return g_last_cuda_error; }

#ifdef TRRT_PHASE_PROF
// experiment builds only: read (and clear) the phase sums of rrt_kernel_spec; synchronises the device
extern "C" int trrt_debug_phase_prof(unsigned long long *host_out24) {
    CUDA_TRY(cudaDeviceSynchronize());
    CUDA_TRY(cudaMemcpyFromSymbol(host_out24, trrt::g_phase_prof, sizeof(unsigned long long) * 24));
    unsigned long long z[24] = {0};
    CUDA_TRY(cudaMemcpyToSymbol(trrt::g_phase_prof, z, sizeof(z)));
    return TRRT_OK;
}
#endif

void trrt_default_params(trrt_params *p) {
    p->thetastar = 1; p->forwardonly = 1; p->bikelength = 5; p->leftconstraint = -65; p->rightconstraint = 65;
    p->frontclearance = 2; p->maxdrivedist = 30; p->tol_xy = 10; p->tol_ang = 45; p->weightxy = .6;
}

size_t trrt_grid_words(int H, int W) { return (size_t)H * (size_t)((W + 31) / 32); }

int trrt_pack_grid(const uint8_t *d_free, int n_maps, int H, int W, uint32_t *d_bits, void *stream) {
    int e = check_map(n_maps, H, W);
    if (e) return e;
    if (!d_free || !d_bits) return TRRT_ERR_INVALID_ARGUMENT;
    int wpr = (W + 31) / 32;
    size_t total = (size_t)n_maps * H * wpr;
    int blocks = (int)((total + 255) / 256);
    if (blocks > sm_count() * 16) blocks = sm_count() * 16;
    pack_grid_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(d_free, n_maps, H, W, wpr, d_bits);
    CUDA_TRY(cudaGetLastError());
    return TRRT_OK;
}

int trrt_los_batch(const uint32_t *d_bits, int n_maps, int H, int W, const int32_t *d_map_id, const int32_t *d_seg, int64_t n,
                   uint8_t *d_out, void *stream) {
    int e = check_map(n_maps, H, W);
    if (e) return e;
    if (n < 0 || !d_bits || (n > 0 && (!d_seg || !d_out))) return TRRT_ERR_INVALID_ARGUMENT;
    if (n == 0) return TRRT_OK;
    if (((uintptr_t)d_seg & 15) != 0) return TRRT_ERR_INVALID_ARGUMENT;
    // One thread per ray (literal Bresenham).  G lanes per ray were measured on the cfg-4 rays (2^20 rays of 1..512 px,
    // 88% blocked): 1 lane 232 us, 8 lanes 231 us, 16 lanes 208 us, 32 lanes 253 us; short clear rays (Theta*) favour 1,
    // and this rows layout is only the comparison arm of the strip kernel (trrt_los_batch_tiled).
    const unsigned blocks = (unsigned)((n + 255) / 256);
    los_batch_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(d_bits, H, W, (W + 31) / 32, d_map_id, (const int4 *)d_seg, n, d_out);
    CUDA_TRY(cudaGetLastError());
    return TRRT_OK;
}

size_t trrt_tile_words(int H, int W) {
    const size_t tp = (size_t)((W > H ? W : H) + 7) / 8;
    return 4 * (tp + 1) * tp; // 2 orientations x (tp+1)*tp entries x 2 uint64
}

int trrt_tile_grid(const uint32_t *d_bits, int n_maps, int H, int W, uint64_t *d_tiles, void *stream) {
    int e = check_map(n_maps, H, W);
    if (e) return e;
    if (!d_bits || !d_tiles || ((uintptr_t)d_tiles & 15) != 0) return TRRT_ERR_INVALID_ARGUMENT;
    const int wpr = (W + 31) / 32, tp = (W + 7) / 8;
    size_t total = (size_t)n_maps * 2 * (tp + 1) * tp;
    int blocks = (int)((total + 255) / 256);
    if (blocks > sm_count() * 16) blocks = sm_count() * 16;
    tile_grid_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(d_bits, n_maps, H, wpr, tp, (uint4 *)d_tiles);
    CUDA_TRY(cudaGetLastError());
    return TRRT_OK;
}

int trrt_los_batch_tiled(const uint64_t *d_tiles, int n_maps, int H, int W, const int32_t *d_map_id, const int32_t *d_seg,
                         int64_t n, uint8_t *d_out, void *stream) {
    int e = check_map(n_maps, H, W);
    if (e) return e;
    if (n < 0 || !d_tiles || (n > 0 && (!d_seg || !d_out))) return TRRT_ERR_INVALID_ARGUMENT;
    if (n == 0) return TRRT_OK;
    if (((uintptr_t)d_seg & 15) != 0 || ((uintptr_t)d_tiles & 15) != 0) return TRRT_ERR_INVALID_ARGUMENT;
    // A warp owns `rpw` consecutive segments (a multiple of 32) and refills idle lanes from them.  The kernel is bound
    // by the integer pipes, not by latency, so long ranges (fewer refill rounds and tails) beat more resident warps:
    // 256 segments per warp when that still gives every SM 24 warps, never fewer than 64.  Measured on the cfg-4 rays:
    // rpw 96 .. 256 -> 73 .. 71 us; refill threshold 6 / 8 / 12 idle lanes -> 72.6 / 70.6 / 70.8 us; cooperative tail
    // from 4 / 8 / 16 remaining rays -> 72.4 / 70.6 / 70.7 us, without it 87 us.
    const int refill_min = 8, coop_max = 8;
    const long long target_warps = (long long)sm_count() * 24;
    long long rpw = ((n + target_warps - 1) / target_warps + 31) / 32 * 32;
    if (rpw < 64) rpw = 64;
    if (rpw > 256) rpw = 256;
    const long long warps = (n + rpw - 1) / rpw;
    const unsigned blocks = (unsigned)((warps + LOS_WARPS - 1) / LOS_WARPS);
    los_tiled_kernel<<<blocks, LOS_WARPS * 32, 0, (cudaStream_t)stream>>>((const uint4 *)d_tiles, H, (W + 7) / 8, d_map_id, (const int4 *)d_seg,
                                                                          (long long)n, (int)rpw, refill_min, coop_max, d_out);
    CUDA_TRY(cudaGetLastError());
    return TRRT_OK;
}

// Launch plan of nearest_batch: TQ queries per warp, `spc` query sets per CTA (the other 8/spc warps of a CTA split
// its node range), grid = (node ranges, set groups).  Slices are multiples of 256 nodes (32 lanes x 2 nodes x 4 loads).
struct NearestPlan {
    int tq, spc_log2, grid_sets, grid_cols, n_slices;
    int64_t slice_len;
};
static NearestPlan nearest_plan(int64_t n_nodes, int64_t n_q) {
    NearestPlan P;
    // as many queries per warp as there are (up to 8): every node load is shared by TQ queries
    P.tq = n_q >= 8 ? 8 : (n_q > 4 ? 8 : (n_q > 2 ? 4 : (n_q > 1 ? 2 : 1)));
    int64_t nsets = (n_q + P.tq - 1) / P.tq;
    P.spc_log2 = 0;
    while ((1 << P.spc_log2) < NN_WARPS && (1 << P.spc_log2) < nsets) P.spc_log2++;
    const int spc = 1 << P.spc_log2, wps = NN_WARPS / spc;
    P.grid_sets = (int)((nsets + spc - 1) / spc);
    // blockIdx.x (fastest in launch order) runs over the set groups, so the CTAs that stream one node range are
    // co-scheduled and share it through L2.  Few set groups = HBM streaming: one wave of 2 CTAs per SM.  Many set
    // groups = fp64 bound: ~8 CTAs per SM in total so that the last wave is nearly full.
    const int per_sm = P.grid_sets <= 2 ? 2 : 8;
    int64_t gx = ((int64_t)sm_count() * per_sm) / P.grid_sets;
    int64_t max_gx = (n_nodes + 512 * (int64_t)wps - 1) / (512 * (int64_t)wps); // at least 512 nodes per warp slice
    if (gx > max_gx) gx = max_gx;
    if (gx > 65535) gx = 65535;
    if (gx < 1) gx = 1;
    int64_t len = (n_nodes + gx * wps - 1) / (gx * wps);
    len = (len + 255) & ~(int64_t)255;
    if (len < 256) len = 256;
    int64_t slices = (n_nodes + len - 1) / len; // slices that hold nodes
    gx = (slices + wps - 1) / wps;
    P.grid_cols = (int)gx;
    P.n_slices = (int)gx; // one partial per CTA column and query (the warps of a set fold their sub-slices in the CTA)
    P.slice_len = len;
    return P;
}

size_t trrt_nearest_workspace_bytes(int64_t n_nodes, int64_t n_q) {
    if (n_nodes <= 0 || n_q <= 0) return 16;
    NearestPlan P = nearest_plan(n_nodes, n_q);
    // [partial d2 | partial index | one arrival counter per query group]
    return (((size_t)P.n_slices * (size_t)n_q * (sizeof(double) + sizeof(int32_t)) + 15) & ~(size_t)15) + (size_t)P.grid_sets * sizeof(unsigned) + 16;
}

int trrt_nearest_batch(const double *d_x, const double *d_y, int64_t n_nodes, const int32_t *d_qxy, int64_t n_q, int32_t *d_idx,
                       double *d_d2, void *d_work, size_t work_bytes, void *stream) {
    if (n_nodes < 0 || n_q < 0 || n_nodes > 0x7ffffffe) return TRRT_ERR_INVALID_ARGUMENT;
    if (n_q == 0) return TRRT_OK;
    if (!d_qxy || !d_idx) return TRRT_ERR_INVALID_ARGUMENT;
    cudaStream_t st = (cudaStream_t)stream;
    if (n_nodes == 0) { // np.argmin([]) raises; report -1
        CUDA_TRY(cudaMemsetAsync(d_idx, 0xff, (size_t)n_q * sizeof(int32_t), st));
        return TRRT_OK;
    }
    if (!d_x || !d_y || !d_work) return TRRT_ERR_INVALID_ARGUMENT;
    if (((uintptr_t)d_x & 15) || ((uintptr_t)d_y & 15) || ((uintptr_t)d_work & 7)) return TRRT_ERR_INVALID_ARGUMENT;
    if (work_bytes < trrt_nearest_workspace_bytes(n_nodes, n_q)) return TRRT_ERR_WORKSPACE_TOO_SMALL;
    const NearestPlan P = nearest_plan(n_nodes, n_q);
    double *part_d = (double *)d_work;
    int32_t *part_i = (int32_t *)(part_d + (size_t)P.n_slices * n_q);
    unsigned *done = (unsigned *)((char *)d_work + (((size_t)P.n_slices * (size_t)n_q * (sizeof(double) + sizeof(int32_t)) + 15) & ~(size_t)15));
    CUDA_TRY(cudaMemsetAsync(done, 0, (size_t)P.grid_sets * sizeof(unsigned), st));
    dim3 grid((unsigned)P.grid_sets, (unsigned)P.grid_cols);
    switch (P.tq) {
    case 8: nearest_tile_kernel<8><<<grid, NN_WARPS * 32, 0, st>>>(d_x, d_y, n_nodes, d_qxy, n_q, P.slice_len, P.spc_log2, part_d, part_i, done, d_idx, d_d2); break;
    case 4: nearest_tile_kernel<4><<<grid, NN_WARPS * 32, 0, st>>>(d_x, d_y, n_nodes, d_qxy, n_q, P.slice_len, P.spc_log2, part_d, part_i, done, d_idx, d_d2); break;
    case 2: nearest_tile_kernel<2><<<grid, NN_WARPS * 32, 0, st>>>(d_x, d_y, n_nodes, d_qxy, n_q, P.slice_len, P.spc_log2, part_d, part_i, done, d_idx, d_d2); break;
    default: nearest_tile_kernel<1><<<grid, NN_WARPS * 32, 0, st>>>(d_x, d_y, n_nodes, d_qxy, n_q, P.slice_len, P.spc_log2, part_d, part_i, done, d_idx, d_d2); break;
    }
    CUDA_TRY(cudaGetLastError());
    return TRRT_OK;
}

static int rrt_tsize(int K) {
    int t = 16;
    while (t < 2 * K) t <<= 1;
    return t;
}
size_t trrt_rrt_workspace_bytes(int64_t n_queries, int32_t K) {
    if (n_queries <= 0 || K <= 0) return 256;
    // [work counter | hash tables]
    return 256 + (size_t)n_queries * (size_t)rrt_tsize(K) * sizeof(int32_t);
}

static BikeParams to_dev(const trrt_params &p) {
    BikeParams b;
    b.thetastar = p.thetastar; b.forwardonly = p.forwardonly; b.bikelength = p.bikelength; b.leftconstraint = p.leftconstraint;
    b.rightconstraint = p.rightconstraint; b.frontclearance = p.frontclearance; b.maxdrivedist = p.maxdrivedist;
    b.tol_xy = p.tol_xy; b.tol_ang = p.tol_ang; b.weightxy = p.weightxy;
    // host evaluation of the device's own rot_make(): bit-identical (trrt_libm.h, no contraction on either side)
    b.r90 = rot_make(90.0); b.rm90 = rot_make(-90.0); b.r180 = rot_make(180.0);
    b.rleft = rot_make(p.leftconstraint); b.rright = rot_make(p.rightconstraint);
    return b;
}

int trrt_rrt_batch(const trrt_rrt_args *args, void *stream) {
    if (!args) return TRRT_ERR_INVALID_ARGUMENT;
    const trrt_rrt_args &A = *args;
    int e = check_map(A.n_maps, A.H, A.W);
    if (e) return e;
    if (A.n_queries < 0 || A.K < 1) return TRRT_ERR_INVALID_ARGUMENT;
    if (A.n_queries == 0) return TRRT_OK;
    if (!A.d_bits || !A.d_start || !A.d_goal || (A.K > 1 && (!A.d_sample_xy || !A.d_sample_th)) || !A.d_node_x || !A.d_node_y || !A.d_node_th ||
        !A.d_parent || !A.d_n_nodes || !A.d_sol || !A.d_status || !A.d_iters || !A.d_work)
        return TRRT_ERR_INVALID_ARGUMENT;
    if (A.d_los_log && !A.d_n_los) return TRRT_ERR_INVALID_ARGUMENT;
    if (A.d_row_start && (!A.d_pack_rows || !A.d_pack_x || !A.d_pack_y || !A.d_pack_th || !A.d_pack_parent || (A.d_pack_u && !A.d_u)))
        return TRRT_ERR_INVALID_ARGUMENT;
    if (A.work_bytes < trrt_rrt_workspace_bytes(A.n_queries, A.K)) return TRRT_ERR_WORKSPACE_TOO_SMALL;
    if ((uintptr_t)A.d_work & 7) return TRRT_ERR_INVALID_ARGUMENT;
    if ((uintptr_t)A.d_sample_xy & (A.sample_xy_i16 ? 3 : 7)) return TRRT_ERR_INVALID_ARGUMENT; // read as short2 / int2
    int G = A.lanes_per_query != 0 ? A.lanes_per_query : 32; // one warp per query unless told otherwise
    RrtDev d;
    d.bits = A.d_bits; d.H = A.H; d.W = A.W; d.wpr = (A.W + 31) / 32; d.map_id = A.d_map_id; d.P = to_dev(A.params);
    d.nq = A.n_queries; d.K = A.K; d.start = A.d_start; d.goal = A.d_goal; d.sxy = (const int32_t *)A.d_sample_xy; d.sxy16 = A.sample_xy_i16 ? 1 : 0; d.sth = A.d_sample_th;
    d.nx = A.d_node_x; d.ny = A.d_node_y; d.nth = A.d_node_th; d.parent = A.d_parent; d.u = A.d_u;
    d.n_nodes = A.d_n_nodes; d.sol = A.d_sol; d.status = A.d_status; d.iters = A.d_iters;
    d.it_near = A.d_it_near; d.it_new = A.d_it_new; d.it_code = A.d_it_code; d.los_log = A.d_los_log; d.n_los = A.d_n_los;
    d.counters = (unsigned long long *)A.d_counters;
    d.next_query = (unsigned long long *)A.d_work;
    d.pack_rows = (unsigned long long *)A.d_pack_rows; d.row_start = (long long *)A.d_row_start;
    d.px = A.d_pack_x; d.py = A.d_pack_y; d.pth = A.d_pack_th; d.pparent = A.d_pack_parent; d.pu = A.d_pack_u;
    d.tab = (int32_t *)((char *)A.d_work + 256); d.tsize = rrt_tsize(A.K);
    cudaStream_t st = (cudaStream_t)stream;
    int threads = 128;
    int64_t blocks = (A.n_queries * G + threads - 1) / threads;
    if (A.schedule == 1) { // cooperative: G lanes on one iteration at a time
        switch (G) {
        case 1: rrt_kernel_coop<1><<<(unsigned)blocks, threads, 0, st>>>(d); break;
        case 2: rrt_kernel_coop<2><<<(unsigned)blocks, threads, 0, st>>>(d); break;
        case 4: rrt_kernel_coop<4><<<(unsigned)blocks, threads, 0, st>>>(d); break;
        case 8: rrt_kernel_coop<8><<<(unsigned)blocks, threads, 0, st>>>(d); break;
        case 16: rrt_kernel_coop<16><<<(unsigned)blocks, threads, 0, st>>>(d); break;
        case 32: rrt_kernel_coop<32><<<(unsigned)blocks, threads, 0, st>>>(d); break;
        default: return TRRT_ERR_INVALID_ARGUMENT;
        }
    } else if (A.schedule == 0) { // speculative window of G iterations, persistent groups
        const size_t smem = 0;
        threads = SPEC_THREADS;
        blocks = (A.n_queries * G + threads - 1) / threads;
        CUDA_TRY(cudaMemsetAsync(d.next_query, 0, sizeof(unsigned long long), st));
        const void *fn = nullptr;
        switch (G) {
        case 1: fn = (const void *)rrt_kernel_spec<1>; break;
        case 2: fn = (const void *)rrt_kernel_spec<2>; break;
        case 4: fn = (const void *)rrt_kernel_spec<4>; break;
        case 8: fn = (const void *)rrt_kernel_spec<8>; break;
        case 16: fn = (const void *)rrt_kernel_spec<16>; break;
        case 32: fn = (const void *)rrt_kernel_spec<32>; break;
        default: return TRRT_ERR_INVALID_ARGUMENT;
        }
        int per_sm = 0;
        CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, threads, smem));
        if (per_sm < 1) per_sm = 1;
        int64_t resident = (int64_t)sm_count() * per_sm; // one full wave; groups loop over the queries
        if (blocks > resident) blocks = resident;
        RrtDev *dp = &d;
        void *kargs[] = {(void *)dp};
        CUDA_TRY(cudaLaunchKernel(fn, dim3((unsigned)blocks), dim3(threads), kargs, smem, st));
    } else return TRRT_ERR_INVALID_ARGUMENT;
    CUDA_TRY(cudaGetLastError());
    return TRRT_OK;
}

int trrt_steer_batch(const trrt_params *params, int64_t n, const double *d_in, double *d_out, uint8_t *d_straight, void *stream) {
    if (!params || n < 0) return TRRT_ERR_INVALID_ARGUMENT;
    if (n == 0) return TRRT_OK;
    if (!d_in || !d_out || !d_straight) return TRRT_ERR_INVALID_ARGUMENT;
    steer_batch_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(to_dev(*params), n, d_in, d_out, d_straight);
    CUDA_TRY(cudaGetLastError());
    return TRRT_OK;
}

int trrt_drive_batch(const trrt_params *params, int64_t n, const double *d_in, double *d_out, void *stream) {
    if (!params || n < 0) return TRRT_ERR_INVALID_ARGUMENT;
    if (n == 0) return TRRT_OK;
    if (!d_in || !d_out) return TRRT_ERR_INVALID_ARGUMENT;
    drive_batch_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(to_dev(*params), n, d_in, d_out);
    CUDA_TRY(cudaGetLastError());
    return TRRT_OK;
}

int trrt_arc_batch(const uint32_t *d_bits, int n_maps, int H, int W, const int32_t *d_map_id, int64_t n, const double *d_in,
                   uint8_t *d_blocked, int lanes, void *stream) {
    int e = check_map(n_maps, H, W);
    if (e) return e;
    if (n < 0) return TRRT_ERR_INVALID_ARGUMENT;
    if (n == 0) return TRRT_OK;
    if (!d_bits || !d_in || !d_blocked) return TRRT_ERR_INVALID_ARGUMENT;
    cudaStream_t st = (cudaStream_t)stream;
    int wpr = (W + 31) / 32;
    if (lanes == 0) lanes = 8;
    int64_t blocks = (n * lanes + 127) / 128;
    switch (lanes) {
    case 1: arc_batch_kernel<1><<<(unsigned)blocks, 128, 0, st>>>(d_bits, H, W, wpr, d_map_id, n, d_in, d_blocked); break;
    case 2: arc_batch_kernel<2><<<(unsigned)blocks, 128, 0, st>>>(d_bits, H, W, wpr, d_map_id, n, d_in, d_blocked); break;
    case 4: arc_batch_kernel<4><<<(unsigned)blocks, 128, 0, st>>>(d_bits, H, W, wpr, d_map_id, n, d_in, d_blocked); break;
    case 8: arc_batch_kernel<8><<<(unsigned)blocks, 128, 0, st>>>(d_bits, H, W, wpr, d_map_id, n, d_in, d_blocked); break;
    case 16: arc_batch_kernel<16><<<(unsigned)blocks, 128, 0, st>>>(d_bits, H, W, wpr, d_map_id, n, d_in, d_blocked); break;
    case 32: arc_batch_kernel<32><<<(unsigned)blocks, 128, 0, st>>>(d_bits, H, W, wpr, d_map_id, n, d_in, d_blocked); break;
    default: return TRRT_ERR_INVALID_ARGUMENT;
    }
    CUDA_TRY(cudaGetLastError());
    return TRRT_OK;
}

int trrt_arc_pixels_batch(int H, int W, int64_t n, const double *d_in, int32_t cap, int32_t *d_pixels, int32_t *d_count, void *stream) {
    int e = check_map(1, H, W);
    if (e) return e;
    if (n < 0 || cap < 0) return TRRT_ERR_INVALID_ARGUMENT;
    if (n == 0) return TRRT_OK;
    if (!d_in || !d_count || (cap > 0 && !d_pixels)) return TRRT_ERR_INVALID_ARGUMENT;
    arc_pixels_kernel<<<(unsigned)((n * 32 + 127) / 128), 128, 0, (cudaStream_t)stream>>>(H, W, n, d_in, cap, d_pixels, d_count);
    CUDA_TRY(cudaGetLastError());
    return TRRT_OK;
}

int trrt_clearance_batch(const uint32_t *d_bits, int n_maps, int H, int W, const int32_t *d_map_id, const trrt_params *params, int64_t n,
                         const double *d_in, uint8_t *d_clear, void *stream) {
    int e = check_map(n_maps, H, W);
    if (e) return e;
    if (!params || n < 0) return TRRT_ERR_INVALID_ARGUMENT;
    if (n == 0) return TRRT_OK;
    if (!d_bits || !d_in || !d_clear) return TRRT_ERR_INVALID_ARGUMENT;
    clearance_batch_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(d_bits, H, W, (W + 31) / 32, d_map_id, to_dev(*params), n,
                                                                                         d_in, d_clear);
    CUDA_TRY(cudaGetLastError());
    return TRRT_OK;
}

int trrt_anglediff_batch(int64_t n, const double *d_in, double *d_out, void *stream) {
    if (n < 0) return TRRT_ERR_INVALID_ARGUMENT;
    if (n == 0) return TRRT_OK;
    if (!d_in || !d_out) return TRRT_ERR_INVALID_ARGUMENT;
    anglediff_batch_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(n, d_in, d_out);
    CUDA_TRY(cudaGetLastError());
    return TRRT_OK;
}

int trrt_findnearest_batch(const trrt_params *params, int64_t n_queries, int32_t K, const double *d_node_x, const double *d_node_y,
                           const double *d_node_th, const int32_t *d_n_nodes, const int32_t *d_it_near, const int32_t *d_it_new,
                           const double *d_goal, int32_t *d_best, double *d_best_dist, void *stream) {
    (void)d_n_nodes;
    if (!params || n_queries < 0 || K < 1) return TRRT_ERR_INVALID_ARGUMENT;
    if (n_queries == 0) return TRRT_OK;
    if (!d_node_x || !d_node_y || !d_node_th || !d_it_near || !d_it_new || !d_goal || !d_best || !d_best_dist) return TRRT_ERR_INVALID_ARGUMENT;
    findnearest_kernel<<<(unsigned)n_queries, 128, 0, (cudaStream_t)stream>>>(to_dev(*params), n_queries, K, d_node_x, d_node_y, d_node_th,
                                                                                d_it_near, d_it_new, d_goal, d_best, d_best_dist);
    CUDA_TRY(cudaGetLastError());
    return TRRT_OK;
}

// Launch plan of theta_batch.  Everything is computed in 64 bits: a slot costs H*W cells of 16 B plus heap_cap entries of
// 16 B (default 2*H*W, i.e. 48*H*W bytes per slot), so large maps times many slots reach hundreds of GB -- the caller caps
// n_slots by the memory it can spare (Planner.theta does), and sizes that do not fit an int32 are refused.
static int theta_plan(trrt_theta_args *A, int *G) {
    int g = A->lanes_per_query;
    if (g == 0) g = 32; // measured on map2: a full warp per search is fastest at every batch size (2048 queries: 96 / 163 / 215 ms for 32 / 16 / 8 lanes)
    if (g < 8) g = 8;
    *G = g;
    if (A->H < 1 || A->W < 1) return TRRT_ERR_INVALID_ARGUMENT;
    if (A->n_slots <= 0) {
        // 16 warps per SM; 24 when the batch has more queries than that (measured on map2: 8192 queries 137 ms vs 152 ms)
        int wps = (A->n_queries * g > (int64_t)sm_count() * 16 * 32) ? 24 : 16;
        int64_t resident = (int64_t)sm_count() * wps * 32 / g;
        A->n_slots = (int32_t)(A->n_queries < resident ? (A->n_queries > 0 ? A->n_queries : 1) : resident);
    }
    if (A->heap_cap <= 0) {
        int64_t c = 2ll * A->H * A->W;
        if (c < 4096) c = 4096;
        if (c > 0x7fffffffll) return TRRT_ERR_MAP_TOO_LARGE; // heap positions are int32
        A->heap_cap = (int32_t)c;
    }
    return TRRT_OK;
}
static size_t theta_cells_bytes(const trrt_theta_args *A) { return (size_t)A->n_slots * (size_t)A->H * (size_t)A->W * sizeof(Cell); }
static size_t theta_heap_bytes(const trrt_theta_args *A) { return (size_t)A->n_slots * (size_t)A->heap_cap * sizeof(HeapEnt); }

size_t trrt_theta_workspace_bytes(trrt_theta_args *args) {
    if (!args) return 0;
    int G;
    if (theta_plan(args, &G) != TRRT_OK) return 0; // 0 = this map cannot be planned (trrt_theta_batch reports why)
    return 256 + theta_cells_bytes(args) + theta_heap_bytes(args);
}

int trrt_theta_batch(const trrt_theta_args *args, void *stream) {
    if (!args) return TRRT_ERR_INVALID_ARGUMENT;
    trrt_theta_args A = *args;
    int e = check_map(A.n_maps, A.H, A.W);
    if (e) return e;
    if (A.n_queries < 0) return TRRT_ERR_INVALID_ARGUMENT;
    if (A.n_queries == 0) return TRRT_OK;
    if (!A.d_bits || !A.d_start_goal || !A.d_path_len || !A.d_cost || !A.d_expanded || !A.d_status || !A.d_work) return TRRT_ERR_INVALID_ARGUMENT;
    if (A.d_path && A.path_cap < 1) return TRRT_ERR_INVALID_ARGUMENT;
    if (A.d_los_log && (A.los_cap < 1 || !A.d_n_los)) return TRRT_ERR_INVALID_ARGUMENT;
    if ((uintptr_t)A.d_work & 15) return TRRT_ERR_INVALID_ARGUMENT;
    int G;
    e = theta_plan(&A, &G);
    if (e) return e;
    if (G != 8 && G != 16 && G != 32) return TRRT_ERR_INVALID_ARGUMENT;
    size_t need = 256 + theta_cells_bytes(&A) + theta_heap_bytes(&A);
    if (A.work_bytes < need) return TRRT_ERR_WORKSPACE_TOO_SMALL;
    cudaStream_t st = (cudaStream_t)stream;
    ThetaDev d;
    d.bits = A.d_bits; d.H = A.H; d.W = A.W; d.wpr = (A.W + 31) / 32; d.map_id = A.d_map_id; d.thetastar = A.thetastar;
    d.nq = A.n_queries; d.sg = A.d_start_goal; d.path = A.d_path; d.path_cap = A.path_cap; d.path_len = A.d_path_len; d.cost = A.d_cost;
    d.expanded = A.d_expanded; d.status = A.d_status; d.los_log = A.d_los_log; d.los_cap = A.los_cap; d.n_los = A.d_n_los;
    d.pushes = A.d_pushes; d.n_slots = A.n_slots; d.heap_cap = A.heap_cap; d.order = A.d_order;
    char *w = (char *)A.d_work;
    d.next_query = (unsigned long long *)w;
    d.cells = (Cell *)(w + 256);
    d.heap = (HeapEnt *)(w + 256 + theta_cells_bytes(&A));
    // stamps must start at epoch 0 (= untouched) and the query counter at 0
    CUDA_TRY(cudaMemsetAsync(w, 0, 256 + theta_cells_bytes(&A), st));
    const int threads = 128;
    int64_t blocks = ((int64_t)A.n_slots * G + threads - 1) / threads;
    switch (G) {
    case 8: theta_kernel<8><<<(unsigned)blocks, threads, 0, st>>>(d); break;
    case 16: theta_kernel<16><<<(unsigned)blocks, threads, 0, st>>>(d); break;
    default: theta_kernel<32><<<(unsigned)blocks, threads, 0, st>>>(d); break;
    }
    CUDA_TRY(cudaGetLastError());
    return TRRT_OK;
}

size_t trrt_mission_workspace_bytes(int64_t n_missions, int32_t K) {
    if (n_missions <= 0 || K < 1) return 256;
    const size_t n = (size_t)n_missions, k = (size_t)K;
    return 19 * 256 + n * (104 + 68 * k + 24 * (k - 1)) + trrt_rrt_workspace_bytes(n_missions, K);
}

int trrt_mission_batch(const trrt_mission_args *args, void *stream) {
    if (!args) return TRRT_ERR_INVALID_ARGUMENT;
    const trrt_mission_args &A = *args;
    int e = check_map(A.n_maps, A.H, A.W);
    if (e) return e;
    if (A.n_missions < 0 || A.K < 2 || A.n_stages < 0 || A.seg_cap < 0 || A.wp_cap < 1 || A.path_cap < 0) return TRRT_ERR_INVALID_ARGUMENT;
    if (A.n_missions == 0) return TRRT_OK;
    if (!A.d_bits || !A.d_waypoints || !A.d_n_waypoints || !A.d_normals || !A.d_normal_range || !A.d_order || (A.n_stages > 0 && !A.n_active) ||
        !A.d_status || !A.d_stop_seg || !A.d_n_seg || !A.d_path_len || (A.path_cap > 0 && (!A.d_path || !A.d_path_seg)) || !A.d_work)
        return TRRT_ERR_INVALID_ARGUMENT;
    if (A.seg_cap > 0 && (!A.d_seg_begin || !A.d_seg_end || !A.d_seg_solution || !A.d_seg_nearest || !A.d_seg_mindist || !A.d_seg_n_nodes ||
                          !A.d_seg_n_edges || !A.d_seg_iters || !A.d_seg_status))
        return TRRT_ERR_INVALID_ARGUMENT;
    if (A.n_stages > A.seg_cap) return TRRT_ERR_INVALID_ARGUMENT;
    for (int s = 0; s < A.n_stages; s++) // the active missions of a stage are a prefix of the slots of the one before
        if (A.n_active[s] < 0 || A.n_active[s] > (s ? A.n_active[s - 1] : A.n_missions)) return TRRT_ERR_INVALID_ARGUMENT;
    if ((uintptr_t)A.d_work & 255) return TRRT_ERR_INVALID_ARGUMENT;
    if (A.work_bytes < trrt_mission_workspace_bytes(A.n_missions, A.K)) return TRRT_ERR_WORKSPACE_TOO_SMALL;
    MissionDev d;
    d.H = A.H; d.W = A.W; d.map_id = A.d_map_id; d.P = to_dev(A.params); d.xystdv = A.xystdv; d.anglestdv = A.anglestdv;
    d.n = A.n_missions; d.K = A.K; d.wp = A.d_waypoints; d.wp_cap = A.wp_cap; d.n_wp = A.d_n_waypoints; d.route_status = A.d_route_status;
    d.normals = A.d_normals; d.nrange = A.d_normal_range; d.order = A.d_order;
    d.seg_cap = A.seg_cap; d.seg_begin = A.d_seg_begin; d.seg_end = A.d_seg_end; d.seg_solution = A.d_seg_solution;
    d.seg_nearest = A.d_seg_nearest; d.seg_mindist = A.d_seg_mindist; d.seg_n_nodes = A.d_seg_n_nodes; d.seg_n_edges = A.d_seg_n_edges;
    d.seg_iters = A.d_seg_iters; d.seg_status = A.d_seg_status;
    d.status = A.d_status; d.stop_seg = A.d_stop_seg; d.n_seg = A.d_n_seg; d.path = A.d_path; d.path_seg = A.d_path_seg;
    d.path_cap = A.path_cap; d.path_len = A.d_path_len;
    const size_t rrt_off = mission_carve(d, A.d_work, A.n_missions, A.K);
    cudaStream_t st = (cudaStream_t)stream;
    int64_t ib = (A.n_missions + MISSION_THREADS - 1) / MISSION_THREADS;
    if (ib > (int64_t)sm_count() * 16) ib = (int64_t)sm_count() * 16;
    mission_init_kernel<<<(unsigned)ib, MISSION_THREADS, 0, st>>>(d);
    CUDA_TRY(cudaGetLastError());
    trrt_rrt_args r;
    memset(&r, 0, sizeof(r));
    r.d_bits = A.d_bits; r.n_maps = A.n_maps; r.H = A.H; r.W = A.W; r.d_map_id = A.d_map_id ? d.q_map : nullptr; r.params = A.params;
    r.K = A.K; r.d_start = d.q_start; r.d_goal = d.q_goal; r.d_sample_xy = d.q_sxy; r.d_sample_th = d.q_sth;
    r.d_node_x = d.nx; r.d_node_y = d.ny; r.d_node_th = d.nth; r.d_parent = d.parent; r.d_u = d.u;
    r.d_n_nodes = d.q_n_nodes; r.d_sol = d.q_sol; r.d_status = d.q_status; r.d_iters = d.q_iters;
    r.d_it_near = d.it_near; r.d_it_new = d.it_new;
    r.d_work = (char *)A.d_work + rrt_off;
    r.work_bytes = A.work_bytes - rrt_off;
    for (int s = 0; s < A.n_stages; s++) {
        const int na = A.n_active[s];
        if (na == 0) break;
        mission_stage_kernel<<<(unsigned)na, MISSION_THREADS, 0, st>>>(d, s);
        CUDA_TRY(cudaGetLastError());
        r.n_queries = na; // slots are a prefix: the per-slot arrays and the RRT workspace of n_missions queries cover it
        e = trrt_rrt_batch(&r, stream);
        if (e) return e;
        mission_commit_kernel<<<(unsigned)na, MISSION_THREADS, 0, st>>>(d, s);
        CUDA_TRY(cudaGetLastError());
    }
    return TRRT_OK;
}

size_t trrt_legacy_normals_workspace_bytes(int64_t n_seeds) { return 256; }

static int legacy_normals_check(const trrt_legacy_normals_args *args) {
    if (!args) return TRRT_ERR_INVALID_ARGUMENT;
    const trrt_legacy_normals_args &A = *args;
    if (A.n_seeds < 0 || A.fix_cap < 0 || !A.d_fix_count) return TRRT_ERR_INVALID_ARGUMENT;
    if (A.n_seeds > 0 && (!A.d_seeds || !A.d_range || !A.d_out || !A.d_work)) return TRRT_ERR_INVALID_ARGUMENT;
    if (A.fix_cap > 0 && (!A.d_fix_pos || !A.d_fix_r2)) return TRRT_ERR_INVALID_ARGUMENT;
    return TRRT_OK;
}

int trrt_legacy_normals_draw(const trrt_legacy_normals_args *args, void *stream) {
    int e = legacy_normals_check(args);
    if (e) return e;
    const trrt_legacy_normals_args &A = *args;
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaMemsetAsync(A.d_fix_count, 0, sizeof(uint64_t), st));
    if (A.n_seeds == 0) return TRRT_OK;
    if ((uintptr_t)A.d_work & 255) return TRRT_ERR_INVALID_ARGUMENT;
    if (A.work_bytes < trrt_legacy_normals_workspace_bytes(A.n_seeds)) return TRRT_ERR_WORKSPACE_TOO_SMALL;
    CUDA_TRY(cudaMemsetAsync(A.d_work, 0, sizeof(unsigned long long), st));
    LegacyNormalsDev d;
    d.n = A.n_seeds; d.seeds = A.d_seeds; d.range = A.d_range; d.out = A.d_out;
    d.fix_pos = A.d_fix_pos; d.fix_r2 = A.d_fix_r2; d.fix_cap = A.fix_cap;
    d.fix_count = (unsigned long long *)A.d_fix_count; d.next = (unsigned long long *)A.d_work;
    int64_t blocks = (A.n_seeds + RNG_WARPS - 1) / RNG_WARPS;
    if (blocks > (int64_t)sm_count() * 8) blocks = (int64_t)sm_count() * 8;
    legacy_normals_kernel<<<(unsigned)blocks, RNG_WARPS * 32, 0, st>>>(d);
    CUDA_TRY(cudaGetLastError());
    return TRRT_OK;
}

int trrt_libm_log_batch(const double *h_in, double *h_out, int64_t n) {
    if (n < 0 || (n > 0 && (!h_in || !h_out))) return TRRT_ERR_INVALID_ARGUMENT;
    // the host's own libm log, on a few threads: the values are independent
    const int64_t per = 1 << 16;
    int nt = (int)std::min<int64_t>((n + per - 1) / per, (int64_t)std::max(1u, std::min(16u, std::thread::hardware_concurrency())));
    auto run = [=](int64_t lo, int64_t hi) {
        for (int64_t i = lo; i < hi; i++) h_out[i] = log(h_in[i]);
    };
    if (nt <= 1) {
        run(0, n);
        return TRRT_OK;
    }
    std::vector<std::thread> th;
    for (int t = 1; t < nt; t++) th.emplace_back(run, n * t / nt, n * (t + 1) / nt);
    run(0, n / nt);
    for (auto &x : th) x.join();
    return TRRT_OK;
}

int trrt_legacy_normals_fixup(const trrt_legacy_normals_args *args, const double *d_fix_log, int64_t n_fix, void *stream) {
    int e = legacy_normals_check(args);
    if (e) return e;
    const trrt_legacy_normals_args &A = *args;
    if (n_fix < 0 || n_fix > A.fix_cap || (n_fix > 0 && !d_fix_log)) return TRRT_ERR_INVALID_ARGUMENT;
    if (n_fix == 0) return TRRT_OK;
    int64_t blocks = (n_fix + 255) / 256;
    if (blocks > (int64_t)sm_count() * 16) blocks = (int64_t)sm_count() * 16;
    legacy_normals_fixup_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(A.d_out, A.d_fix_pos, A.d_fix_r2, d_fix_log, n_fix);
    CUDA_TRY(cudaGetLastError());
    return TRRT_OK;
}

int trrt_rand_conf_batch(int H, int W, double xystdv, double anglestdv, int64_t n, int32_t n_samples, const double *d_goal,
                         const double *d_normals, void *d_sample_xy, int32_t sample_xy_i16, double *d_sample_th, void *stream) {
    if (H < 1 || W < 1 || n < 0 || n_samples < 0) return TRRT_ERR_INVALID_ARGUMENT;
    if (sample_xy_i16 && (H > 32768 || W > 32768)) return TRRT_ERR_MAP_TOO_LARGE;
    const int64_t total = n * (int64_t)n_samples;
    if (total == 0) return TRRT_OK;
    if (!d_goal || !d_normals || !d_sample_xy || !d_sample_th) return TRRT_ERR_INVALID_ARGUMENT;
    int64_t blocks = (total + 255) / 256;
    if (blocks > (int64_t)sm_count() * 16) blocks = (int64_t)sm_count() * 16;
    cudaStream_t st = (cudaStream_t)stream;
    if (sample_xy_i16)
        rand_conf_kernel<int16_t><<<(unsigned)blocks, 256, 0, st>>>(H, W, xystdv, anglestdv, n, n_samples, d_goal, d_normals,
                                                                    (int16_t *)d_sample_xy, d_sample_th);
    else
        rand_conf_kernel<int32_t><<<(unsigned)blocks, 256, 0, st>>>(H, W, xystdv, anglestdv, n, n_samples, d_goal, d_normals,
                                                                    (int32_t *)d_sample_xy, d_sample_th);
    CUDA_TRY(cudaGetLastError());
    return TRRT_OK;
}

} // extern "C"
