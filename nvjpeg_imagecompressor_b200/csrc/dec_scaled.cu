// dec_scaled.cu -- reduced-size decode (libjpeg's DCT scaling, scale_num = 1, scale_denom = 2 / 4 / 8): one inverse DCT
// per block that writes S x S samples (S = 8 / denom) instead of 8 x 8, so a 1/8 decode writes 1/64 of the pixels.
// The entropy stages and the DC prefix sums are the full-size decoder's; only the back end changes:
//   k_idct_scaled  de-quantise + jidctred.c jpeg_idct_1x1 / 2x2 / 4x4 (jidctint.c islow for 8 x 8), one thread per block
//   k_upcolor      unchanged, on a Geom that describes the scaled planes (dec_kernels.h dec_scale_setup)
// Blocks whose output is one sample are their DC alone: they read the compact DC array (2 bytes) and no coefficients.
#include <algorithm>

#include "common.cuh"
#include "dec.h"
#include "dec_idct.cuh"
#include "dec_kernels.h"

namespace b2j {

constexpr int SC_THREADS = 256;

__device__ __forceinline__ uint8_t clamp_sample(int v) { return (uint8_t)min(255, max(0, v + 128)); }

// jidctred.c jpeg_idct_2x2: columns / rows 0, 1, 3, 5, 7 only; x is de-quantised, natural order
__device__ __forceinline__ void idct2x2(const int (&x)[64], uint8_t (&o)[64]) {
    int ws[16];
#pragma unroll
    for (int c = 0; c < 8; c++) {
        if (c == 2 || c == 4 || c == 6) continue;
        const int t10 = x[c] << 15;
        const int t0 = -5906 * x[56 + c] + 6967 * x[40 + c] - 10426 * x[24 + c] + 29692 * x[8 + c];
        ws[c] = (t10 + t0 + (1 << 12)) >> 13;
        ws[8 + c] = (t10 - t0 + (1 << 12)) >> 13;
    }
#pragma unroll
    for (int r = 0; r < 2; r++) {
        const int *w = ws + 8 * r;
        const int t10 = w[0] << 15;
        const int t0 = -5906 * w[7] + 6967 * w[5] - 10426 * w[3] + 29692 * w[1];
        o[2 * r] = clamp_sample((t10 + t0 + (1 << 19)) >> 20);
        o[2 * r + 1] = clamp_sample((t10 - t0 + (1 << 19)) >> 20);
    }
}

// jidctred.c jpeg_idct_4x4: row / column 4 is never read; pass 1 descales by 12, pass 2 by 19
template <int SH>
__device__ __forceinline__ void idct4(int i0, int i1, int i2, int i3, int i5, int i6, int i7, int (&o)[4]) {
    constexpr int RND = 1 << (SH - 1);
    const int t0e = i0 << 14, t2e = 15137 * i2 - 6270 * i6;
    const int t10 = t0e + t2e, t12 = t0e - t2e;
    const int t0 = -1730 * i7 + 11893 * i5 - 17799 * i3 + 8697 * i1;
    const int t2 = -4176 * i7 - 4926 * i5 + 7373 * i3 + 20995 * i1;
    o[0] = (t10 + t2 + RND) >> SH; o[1] = (t12 + t0 + RND) >> SH;
    o[2] = (t12 - t0 + RND) >> SH; o[3] = (t10 - t2 + RND) >> SH;
}
__device__ __forceinline__ void idct4x4(const int (&x)[64], uint8_t (&o)[64]) {
    int ws[32];
#pragma unroll
    for (int c = 0; c < 8; c++) {
        if (c == 4) continue;
        int t[4];
        idct4<12>(x[c], x[8 + c], x[16 + c], x[24 + c], x[40 + c], x[48 + c], x[56 + c], t);
#pragma unroll
        for (int r = 0; r < 4; r++) ws[r * 8 + c] = t[r];
    }
#pragma unroll
    for (int r = 0; r < 4; r++) {
        const int *w = ws + 8 * r;
        int t[4];
        idct4<19>(w[0], w[1], w[2], w[3], w[5], w[6], w[7], t);
#pragma unroll
        for (int c = 0; c < 4; c++) o[r * 4 + c] = clamp_sample(t[c]);
    }
}

__device__ __forceinline__ void idct8x8(int (&v)[64], uint8_t (&o)[64]) {
#pragma unroll
    for (int c = 0; c < 8; c++) idct8<11>(v[c], v[8 + c], v[16 + c], v[24 + c], v[32 + c], v[40 + c], v[48 + c], v[56 + c]);
#pragma unroll
    for (int r = 0; r < 8; r++) {
        idct8<18>(v[r * 8], v[r * 8 + 1], v[r * 8 + 2], v[r * 8 + 3], v[r * 8 + 4], v[r * 8 + 5], v[r * 8 + 6], v[r * 8 + 7]);
#pragma unroll
        for (int c = 0; c < 8; c++) o[r * 8 + c] = clamp_sample(v[r * 8 + c]);
    }
}

// K x K samples of one block into o (row-major, K per row). sc: the block's 128 coefficient bytes in shared memory,
// chunk c at sc[c ^ sw] (K > 1 only); q: natural-order de-quantisation table; dcv: the un-differenced DC
template <int K>
__device__ __forceinline__ void block_samples(const uint4 *sc, int sw, const int *q, int dcv, uint8_t (&o)[64]) {
    if (K == 1) {
        o[0] = clamp_sample((dcv * q[0] + 4) >> 3);
        return;
    }
    int x[64];
#pragma unroll
    for (int ch = 0; ch < 8; ch++) {
        const uint4 w = sc[ch ^ sw];
        const uint32_t ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
        for (int j = 0; j < 8; j++) {
            const int n = zigzag_nat(ch * 8 + j);
            const int cv = (j & 1) ? ((int)ww[j >> 1] >> 16) : (int)(int16_t)(ww[j >> 1] & 0xFFFFu);
            x[n] = cv * q[n];
        }
    }
    x[0] = dcv * q[0];
    if (K == 2) idct2x2(x, o);
    else if (K == 4) idct4x4(x, o);
    else idct8x8(x, o);
}

// K x K samples to a plane of pitch `stride` (rows of K bytes; dst is K-aligned: the planes are 64-byte aligned and
// their pitches multiples of 8)
template <int K>
__device__ __forceinline__ void store_plane(uint8_t *dst, size_t stride, const uint8_t (&o)[64]) {
#pragma unroll
    for (int r = 0; r < K; r++) {
        uint8_t *d = dst + r * stride;
        if (K == 1) {
            d[0] = o[0];
        } else if (K == 2) {
            *reinterpret_cast<uint16_t *>(d) = (uint16_t)(o[2 * r] | (o[2 * r + 1] << 8));
        } else if (K == 4) {
            *reinterpret_cast<uint32_t *>(d) = (uint32_t)o[4 * r] | ((uint32_t)o[4 * r + 1] << 8) |
                                               ((uint32_t)o[4 * r + 2] << 16) | ((uint32_t)o[4 * r + 3] << 24);
        } else {
            uint32_t lo = 0, hi = 0;
#pragma unroll
            for (int c = 0; c < 4; c++) { lo |= (uint32_t)o[8 * r + c] << (8 * c); hi |= (uint32_t)o[8 * r + 4 + c] << (8 * c); }
            *reinterpret_cast<uint2 *>(d) = make_uint2(lo, hi);
        }
    }
}

// One thread per block, persistent CTAs; every warp takes 32 consecutive blocks at a time and loads the coefficients of
// those that need them (output size above 1) with coalesced 16-byte loads into its own bank-swizzled shared slice.
// g: the file's block layout; v: the scaled view (dec_scale_setup): output size v.W x v.H, Y plane pitch
// v.mcux * 8 * v.hs, chroma pitch v.mcux * 8.
// S / SC: output size of a luma / chroma block. GRAY: luma only, straight into the caller's pitched image, clipped at
// v.W / v.H. REP (SC = 1 only): 1 = every chroma sample stored twice side by side, 2 = twice one above the other (the
// plain replication libjpeg does for 4:2:2 / 4:4:0 at 1/8, where its fancy filters are off).
template <int S, int SC, bool GRAY, int REP>
__global__ void __launch_bounds__(SC_THREADS)
k_idct_scaled(const int16_t *__restrict__ coef, const int16_t *__restrict__ dcarr, Geom g, Geom v, const DecTables *__restrict__ tb,
              uint8_t *__restrict__ py, uint8_t *__restrict__ pcb, uint8_t *__restrict__ pcr, int rst_mcus, size_t out_step) {
    constexpr bool LOAD = S > 1 || (!GRAY && SC > 1);   // some block needs more than its DC
    __shared__ __align__(16) uint4 s_c[LOAD ? SC_THREADS * 8 : 1];
    __shared__ int s_q[2][64];                       // natural order
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid < 128) s_q[tid >> 6][tid & 63] = (int)tb->q[tid >> 6][tid & 63];
    __syncthreads();
    const int hv = GRAY ? g.hs * g.vs : g.bpm - 2;   // luma blocks per MCU (a colour file on a gray context keeps its chroma)
    const size_t ys = (size_t)v.mcux * 8 * v.hs, cs = (size_t)v.mcux * 8;
    uint4 *sw = s_c + (LOAD ? warp * 32 * 8 : 0);
    const uint4 *coef4 = reinterpret_cast<const uint4 *>(coef);
    // the block needs its coefficients (not only its DC): a luma block if S > 1, a chroma block if SC > 1
    auto wants = [&](int b) {
        const int bn = b % g.bpm;
        return bn < hv ? S > 1 : (!GRAY && SC > 1);
    };
    for (int base = (blockIdx.x * (SC_THREADS / 32) + warp) * 32; base < g.nblocks; base += gridDim.x * SC_THREADS) {
        if (LOAD) {
            __syncwarp();   // the slice's previous blocks are done
#pragma unroll
            for (int i = 0; i < 8; i++) {
                const int k = i * 32 + lane, bl = k >> 3, c = k & 7, b = base + bl;
                if (b < g.nblocks && wants(b)) sw[bl * 8 + (c ^ (bl & 7))] = __ldg(coef4 + (size_t)b * 8 + c);
            }
            __syncwarp();
        }
        const int b = base + lane;
        if (b >= g.nblocks) continue;
        const int m = b / g.bpm, bn = b - m * g.bpm;
        if (GRAY && bn >= hv) continue;
        const int my = m / g.mcux, mx = m - my * g.mcux;
        const bool isY = bn < hv;
        // the un-differenced DC, as k_idct takes it: k_dc_scan's running sum from the start of the block's restart
        // interval, or (dcarr == NULL: progressive files) the coefficient array's own DC
        int dcv = dcarr ? (int)dcarr[b] : (int)coef[(size_t)b * 64];
        if (dcarr && rst_mcus > 0 && m >= rst_mcus) {
            const int pm = (m / rst_mcus) * rst_mcus - 1;   // last MCU of the previous interval
            dcv = (int16_t)(dcv - (int)dcarr[pm * g.bpm + (isY ? hv - 1 : bn)]);
        }
        const int *q = s_q[isY ? 0 : 1];
        const uint4 *sc = sw + lane * 8;
        uint8_t o[64];
        if (isY) {
            block_samples<S>(sc, lane & 7, q, dcv, o);
            const int by = bn / g.hs, bx = bn - by * g.hs;
            const int gy0 = (my * g.vs + by) * S, gx0 = (mx * g.hs + bx) * S;
            if (GRAY) {
                const int nr = min(S, v.H - gy0), ncol = min(S, v.W - gx0);
                uint8_t *dst = py + (size_t)gy0 * out_step + gx0;
                for (int r = 0; r < nr; r++)
                    for (int c = 0; c < ncol; c++) dst[(size_t)r * out_step + c] = o[r * S + c];
            } else {
                store_plane<S>(py + (size_t)gy0 * ys + gx0, ys, o);
            }
        } else if (!GRAY) {
            block_samples<SC>(sc, lane & 7, q, dcv, o);
            uint8_t *pl = bn == hv ? pcb : pcr;
            if (REP == 1) {
                pl[(size_t)my * cs + 2 * mx] = o[0];
                pl[(size_t)my * cs + 2 * mx + 1] = o[0];
            } else if (REP == 2) {
                pl[(size_t)(2 * my) * cs + mx] = o[0];
                pl[(size_t)(2 * my + 1) * cs + mx] = o[0];
            } else {
                store_plane<SC>(pl + (size_t)my * SC * cs + (size_t)mx * SC, cs, o);
            }
        }
    }
}

template <int S, int SC, bool GRAY, int REP>
static cudaError_t scaled_one(const int16_t *coef, const int16_t *dcarr, const Geom &g, const Geom &v, const void *tb, uint8_t *py,
                              uint8_t *pcb, uint8_t *pcr, int rst_mcus, size_t out_step, cudaStream_t s) {
    const int nwarps = (g.nblocks + 31) / 32;
    const int grid = std::max(1, std::min((nwarps + SC_THREADS / 32 - 1) / (SC_THREADS / 32), 148 * 4));
    k_idct_scaled<S, SC, GRAY, REP><<<grid, SC_THREADS, 0, s>>>(coef, dcarr, g, v, (const DecTables *)tb, py, pcb, pcr, rst_mcus, out_step);
    return cudaGetLastError();
}

cudaError_t launch_idct_scaled(const int16_t *coef, const int16_t *dcarr, const Geom &g, const DecScale &sc, const void *tb,
                               uint8_t *py, uint8_t *pcb, uint8_t *pcr, bool gray, size_t out_step, int rst_mcus, cudaStream_t s) {
    const Geom &v = sc.view;
    if (gray) {
        if (sc.S == 4) return scaled_one<4, 4, true, 0>(coef, dcarr, g, v, tb, py, nullptr, nullptr, rst_mcus, out_step, s);
        if (sc.S == 2) return scaled_one<2, 2, true, 0>(coef, dcarr, g, v, tb, py, nullptr, nullptr, rst_mcus, out_step, s);
        if (sc.S == 1) return scaled_one<1, 1, true, 0>(coef, dcarr, g, v, tb, py, nullptr, nullptr, rst_mcus, out_step, s);
        return cudaErrorInvalidValue;
    }
    const int key = sc.S * 100 + sc.Sc * 10 + sc.rep;
    switch (key) {
    case 440: return scaled_one<4, 4, false, 0>(coef, dcarr, g, v, tb, py, pcb, pcr, rst_mcus, 0, s);
    case 480: return scaled_one<4, 8, false, 0>(coef, dcarr, g, v, tb, py, pcb, pcr, rst_mcus, 0, s);
    case 220: return scaled_one<2, 2, false, 0>(coef, dcarr, g, v, tb, py, pcb, pcr, rst_mcus, 0, s);
    case 240: return scaled_one<2, 4, false, 0>(coef, dcarr, g, v, tb, py, pcb, pcr, rst_mcus, 0, s);
    case 110: return scaled_one<1, 1, false, 0>(coef, dcarr, g, v, tb, py, pcb, pcr, rst_mcus, 0, s);
    case 111: return scaled_one<1, 1, false, 1>(coef, dcarr, g, v, tb, py, pcb, pcr, rst_mcus, 0, s);
    case 112: return scaled_one<1, 1, false, 2>(coef, dcarr, g, v, tb, py, pcb, pcr, rst_mcus, 0, s);
    case 120: return scaled_one<1, 2, false, 0>(coef, dcarr, g, v, tb, py, pcb, pcr, rst_mcus, 0, s);
    default: return cudaErrorInvalidValue;
    }
}

}  // namespace b2j
