// enc_fdct.cu -- K1: BGR -> YCbCr -> chroma downsample -> islow FDCT -> quantise -> run-length TOKENS in scan order,
// with the symbol histograms (optimized-Huffman pass 1) taken from the compacted tokens.
//
// Replaces the first half of nvjpegEncodeImage (reference call site ImageCompressorImpl.cu:280; nvJPEG kernels
// format_to_ycbcr_kernel / subsample_chroma_kernel / forwardDct32x8Kernel, SURVEY.md 2b). Arithmetic follows
// libjpeg-turbo (jccolor.c, jcsample.c, jfdctint.c, jcdctmgr.c) as restated in SURVEY.md Appendix A.2-A.6,
// bit-exactly (tests/ compare every stage with the CPU checker).
//
// A tile is up to TM_MAX MCUs inside one MCU row; persistent CTAs (up to three per SM) code tile after tile:
//   TMA bulk copies (cp.async.bulk, one per pixel row) stage the raw BGR rows in shared memory   [interior tiles]
//            (issued while the CTA's previous tile is still being coded: before its stage C when its token run
//            leaves the staged rows alone, else after it)
//   stage A: every thread converts 8 pixels x VS rows -> Y / Cb / Cr sample planes in shared memory
//            (gray, NC = 1: the staged rows ARE the Y plane -- jccolor.c grayscale_convert is a copy -- and an MCU is
//            one block, so a tile holds PACK_BLOCKS MCUs: 2048 pixels x 8 rows, the 16 KB of a 4:4:4 tile's rows)
//   stage B: one thread per 8x8 block: 64 samples in registers, both FDCT passes, reciprocal quantisation in place,
//            branch-free count of the non-zero coefficients; a CTA scan of the counts gives every block its place
//            in the tile's token run, then the jchuff.c run-length walk stores one (run | value) entry per non-zero
//            coefficient straight to its final slot of the run in shared memory (two-instruction divergent body)
//   stage C: the whole CTA walks the run in output order: entry -> (ZRL count | table | run/size symbol | value
//            bits), symbol statistics with full-warp shared atomics, coalesced stores to the token pool
// The entropy coder (enc_huff.cu k_pack) then works token-parallel: uniform work per lane instead of a divergent
// per-coefficient branch. With DUMP the quantised coefficients are also written (16-byte stores straight from the
// registers): the parity tests read them, and the secondary-compression path reconstructs the image from them
// (b2j_reconstruct_device: de-quantise + IDCT + upsample, no entropy decode).
#include <algorithm>
#include <atomic>

#include "common.cuh"
#include "kernels.h"

namespace b2j {

template <int HS, int VS, int NC = 3>
struct K1 {
    static_assert(NC == 3 || (NC == 1 && HS == 1 && VS == 1), "gray is one 1x1 component");
    static constexpr int HV = HS * VS;
    static constexpr int BPM = NC == 1 ? 1 : HV + 2;
    static constexpr int TM_MAX = (256 / BPM) & ~1;  // 444: 84, 422/440: 64, 420/411: 42, gray: 256
    static constexpr int MCU_W = 8 * HS, MCU_H = 8 * VS;
    static constexpr int TILE_PX = TM_MAX * MCU_W;
    static constexpr int RAW_STRIDE = TILE_PX * NC;  // multiple of 16 for all six modes
    static constexpr int RAW_BYTES = RAW_STRIDE * MCU_H;
    static constexpr int TOK_BYTES = 64 * 256 * 4 + 256;    // the tile's token run: <= 64 tokens per block
    static constexpr int Y_STRIDE = NC == 1 ? RAW_STRIDE : TILE_PX;
    static constexpr int Y_BYTES = Y_STRIDE * MCU_H;
    static constexpr int C_STRIDE = TM_MAX * 8;
    static constexpr int C_BYTES = C_STRIDE * 8;
    // the staged pixel rows and the sample planes both live inside the token area: the planes are dead before the
    // first token is stored (a barrier separates the sample loads of stage B from its token stores). The planes sit at
    // the front, the staged rows in the last RAW_BYTES: a run of at most OFF_RAW / 4 tokens leaves them untouched, so
    // the next tile's rows can be in flight while such a run is written. Gray: the staged rows are the Y plane.
    static constexpr int OFF_RAW = TOK_BYTES - RAW_BYTES;
    static constexpr int OFF_Y = NC == 1 ? OFF_RAW : 0;
    static constexpr int OFF_CB = OFF_Y + Y_BYTES;
    static constexpr int OFF_CR = OFF_CB + C_BYTES;
    static constexpr int OFF_Q = TOK_BYTES;              // float[3][64] (+ pad): luma, chroma, all-zero (dummy blocks)
    static constexpr int OFF_HIST = OFF_Q + 1536;        // uint32[1024], index = token bits [25:16]
    static constexpr int OFF_DC = OFF_HIST + 4096;       // int16[256]
    static constexpr int OFF_MISC = OFF_DC + 512;        // warp totals[8], pool base, chroma DC token offsets, tile state
    static constexpr int OFF_BAR = OFF_MISC + 64;        // mbarrier
    static constexpr int SMEM = OFF_BAR + 16;
    static_assert(NC == 1 || OFF_CR + C_BYTES <= OFF_RAW, "planes must not overlap the staged rows");
    static_assert(SMEM <= 75 * 1024, "three CTAs per SM");
    static_assert(OFF_RAW >= 0 && OFF_RAW % 16 == 0, "staged rows must fit in the token area, 16-byte aligned");
    static_assert(RAW_STRIDE % 16 == 0, "row stride must allow 16-byte bulk copies");
};

// ---- libjpeg jfdctint.c constants (CONST_BITS = 13) ----
#define FIX_0_298631336 2446
#define FIX_0_390180644 3196
#define FIX_0_541196100 4433
#define FIX_0_765366865 6270
#define FIX_0_899976223 7373
#define FIX_1_175875602 9633
#define FIX_1_501321110 12299
#define FIX_1_847759065 15137
#define FIX_1_961570560 16069
#define FIX_2_053119869 16819
#define FIX_2_562915447 20995
#define FIX_3_072711026 25172

template <bool PASS2>
__device__ __forceinline__ void fdct8(int &d0, int &d1, int &d2, int &d3, int &d4, int &d5, int &d6, int &d7) {
    constexpr int SH = PASS2 ? 15 : 11;
    constexpr int RND = 1 << (SH - 1);
    int t0 = d0 + d7, t7 = d0 - d7, t1 = d1 + d6, t6 = d1 - d6, t2 = d2 + d5, t5 = d2 - d5, t3 = d3 + d4, t4 = d3 - d4;
    int t10 = t0 + t3, t13 = t0 - t3, t11 = t1 + t2, t12 = t1 - t2;
    if (!PASS2) {
        d0 = (t10 + t11) << 2;
        d4 = (t10 - t11) << 2;
    } else {
        d0 = (t10 + t11 + 2) >> 2;
        d4 = (t10 - t11 + 2) >> 2;
    }
    int z1 = (t12 + t13) * FIX_0_541196100;
    d2 = (z1 + t13 * FIX_0_765366865 + RND) >> SH;
    d6 = (z1 - t12 * FIX_1_847759065 + RND) >> SH;
    z1 = t4 + t7;
    int z2 = t5 + t6, z3 = t4 + t6, z4 = t5 + t7;
    int z5 = (z3 + z4) * FIX_1_175875602;
    t4 *= FIX_0_298631336;
    t5 *= FIX_2_053119869;
    t6 *= FIX_3_072711026;
    t7 *= FIX_1_501321110;
    z1 *= -FIX_0_899976223;
    z2 *= -FIX_2_562915447;
    z3 = z3 * (-FIX_1_961570560) + z5;
    z4 = z4 * (-FIX_0_390180644) + z5;
    d7 = (t4 + z1 + z3 + RND) >> SH;
    d5 = (t5 + z2 + z4 + RND) >> SH;
    d3 = (t6 + z2 + z3 + RND) >> SH;
    d1 = (t7 + z1 + z4 + RND) >> SH;
}

// ---- pass 1 (rows) on packed samples. Every jfdctint.c row output is an exact integer combination of the eight
// samples followed by ONE descale, so it can be evaluated as four 2-way dot products (IDP.2A: signed 16-bit
// coefficient pairs x unsigned 8-bit samples) straight on the packed bytes: no unpacking, no butterflies. The
// coefficient matrix below is jfdctint.c's pass 1 applied to unit vectors (CONST_BITS 13, before the descale);
// rows 0 and 4 (coefficients +-4, no descale) take two 4-way dot products each.
__device__ __forceinline__ int dp2a_lo_su(int a, uint32_t b, int c) {
    int d;
    asm("dp2a.lo.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
__device__ __forceinline__ int dp2a_hi_su(int a, uint32_t b, int c) {
    int d;
    asm("dp2a.hi.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
__device__ __forceinline__ uint32_t dp2a_lo_uu(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t d;
    asm("dp2a.lo.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
__device__ __forceinline__ uint32_t dp2a_hi_uu(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t d;
    asm("dp2a.hi.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
__device__ __forceinline__ int dp4a_us(uint32_t a, int b, int c) {
    int d;
    asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
#define B2J_PAIR(lo, hi) ((int)((((uint32_t)(hi)) << 16) | (((uint32_t)(lo)) & 0xFFFFu)))
template <int K>
__device__ __forceinline__ int fdct_row_out(uint32_t x03, uint32_t x47) {
    constexpr int M[8][8] = {{4, 4, 4, 4, 4, 4, 4, 4},
                             {11363, 9633, 6437, 2260, -2260, -6437, -9633, -11363},
                             {10703, 4433, -4433, -10703, -10703, -4433, 4433, 10703},
                             {9633, -2259, -11362, -6436, 6436, 11362, 2259, -9633},
                             {4, -4, -4, 4, 4, -4, -4, 4},
                             {6437, -11362, 2261, 9633, -9633, -2261, 11362, -6437},
                             {4433, -10704, 10704, -4433, -4433, 10704, -10704, 4433},
                             {2260, -6436, 9633, -11363, 11363, -9633, 6436, -2260}};
    if (K == 0) return dp4a_us(x47, 0x04040404, dp4a_us(x03, 0x04040404, 0));
    if (K == 4) return dp4a_us(x47, 0x04FCFC04, dp4a_us(x03, 0x04FCFC04, 0));
    int a = 1024;   // DESCALE(x, CONST_BITS - PASS1_BITS) rounding
    a = dp2a_lo_su(B2J_PAIR(M[K][0], M[K][1]), x03, a);
    a = dp2a_hi_su(B2J_PAIR(M[K][2], M[K][3]), x03, a);
    a = dp2a_lo_su(B2J_PAIR(M[K][4], M[K][5]), x47, a);
    a = dp2a_hi_su(B2J_PAIR(M[K][6], M[K][7]), x47, a);
    return a >> 11;
}
template <int K>
__device__ __forceinline__ void fdct_rows_k(const uint32_t (&xin)[16], int (&v)[64]) {
#pragma unroll
    for (int r = 0; r < 8; r++) v[r * 8 + K] = fdct_row_out<K>(xin[2 * r], xin[2 * r + 1]);
}

// jccolor.c rgb_ycc_convert, 16-bit fixed point
__device__ __forceinline__ void ycc(int b, int g, int r, int &y, int &cb, int &cr) {
    y = (19595 * r + 38470 * g + 7471 * b + 32768) >> 16;
    cb = (-11059 * r - 21709 * g + 32768 * b + ((128 << 16) + 32767)) >> 16;
    cr = (32768 * r - 27439 * g - 5329 * b + ((128 << 16) + 32767)) >> 16;
}

__device__ __forceinline__ int nbits_of(int v) { return 32 - __clz(v < 0 ? -v : v); }

// Stage C of k_fdct: entries (run and table fields as in the final token | coefficient, DC difference or 0 for EOB)
// become final tokens (common.cuh) with ONE formula for DC, AC and EOB entries: the size is the bit length of |value|,
// the value bits are jchuff.c's (value, or value - 1 if negative, masked). Raw-DC tokens (first MCU of the tile) pass
// through. Every token counts one symbol in the bin given by its bits [25:16]; the three raw-DC tokens land in bins
// 2 / 7 / 11 and are taken out again by thread 0 (k_dc_edge_hist counts their real symbols).
template <bool HIST, int NC>
__device__ __forceinline__ void stage_c(const uint32_t *tok, uint32_t *__restrict__ dst, uint32_t total, uint32_t *hs, int tid) {
#pragma unroll 4
    for (uint32_t i = tid; i < total; i += 256) {
        const uint32_t e = tok[i];
        const int z = (int)(int16_t)(e & 0xFFFFu);
        uint32_t msb;
        asm("bfind.u32 %0, %1;" : "=r"(msb) : "r"((uint32_t)abs(z)));
        const uint32_t nb = msb + 1u;           // bfind(0) = -1
        const uint32_t vb = (uint32_t)(z + (z >> 31)) & ((1u << nb) - 1u);
        const uint32_t conv = (e & 0x0FC30000u) | (nb << 18) | vb;   // the walk's carries into the size field go away here
        const uint32_t tk = (e & TOK_RAWDC) ? e : conv;
        dst[i] = tk;
        if (HIST) {
            atomicAdd(&hs[(tk >> 16) & 0x3FFu], 1u);
            const uint32_t nz = (tk >> 26) & 3u;        // ZRL (0xF0) symbols ahead of this coefficient: about one token in sixty
            // bin of the ZRL symbol of this token's AC table: run 15, size 0, table field (tcode + 15) & 3 = (field - run - 1) & 3
            if (nz) atomicAdd(&hs[(15u << 6) | (((tk >> 16) - (tk >> 22) - 1u) & 3u)], nz);
        }
    }
    if (HIST && tid == 0) {   // tcode 2 / 3 | component << 2
        atomicSub(&hs[2], 1u);
        if (NC == 3) { atomicSub(&hs[7], 1u); atomicSub(&hs[11], 1u); }
    }
}

__device__ __forceinline__ uint32_t ld_volatile_shared(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.volatile.shared.u32 %0, [%1];" : "=r"(v) : "r"(smem_u32(p)));
    return v;
}

// Position of tile t (0-based inside a launch that starts at MCU row my0) and whether its pixels need no padding.
struct TilePos {
    int my, tx, mx0, nmcu, x0, y0, tile_px;
    bool interior;
};
template <int MCU_W, int MCU_H>
__device__ __forceinline__ TilePos tile_pos(const Geom &g, int my0, int t) {
    TilePos p;
    const int ty = t / g.tiles_x;
    p.tx = t - ty * g.tiles_x;
    p.my = my0 + ty;
    p.mx0 = p.tx * g.tm;
    p.nmcu = min(g.tm, g.mcux - p.mx0);
    p.x0 = p.mx0 * MCU_W;
    p.y0 = p.my * MCU_H;
    p.tile_px = p.nmcu * MCU_W;
    p.interior = (p.x0 + p.tile_px <= g.W) && (p.y0 + MCU_H <= g.H);
    return p;
}

// Thread 0: one bulk copy per pixel row of tile t into the staged-row region, completing on `bar`. Only interior tiles
// of a launch with bulk_ok are staged this way; the caller waits on the barrier under the same condition.
template <int HS, int VS, int NC>
__device__ __forceinline__ void stage_rows(const uint8_t *img, size_t step, const Geom &g, int my0, int t, int ntl,
                                           uint8_t *raw, uint64_t *bar) {
    using C = K1<HS, VS, NC>;
    if (t >= ntl) return;
    const TilePos p = tile_pos<C::MCU_W, C::MCU_H>(g, my0, t);
    if (!p.interior) return;
    const unsigned row_bytes = (unsigned)p.tile_px * NC;
    const uint8_t *src = img + (size_t)p.y0 * step + (size_t)p.x0 * NC;
    // the CTA's generic-proxy reads and writes of the region (earlier tiles) come before these async-proxy writes
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    mbar_expect_tx(bar, row_bytes * C::MCU_H);
#pragma unroll
    for (int r = 0; r < C::MCU_H; r++) bulk_g2s(raw + r * C::RAW_STRIDE, src + (size_t)r * step, row_bytes, bar);
}

// Persistent CTAs: CTA b codes tile b of the launch's ntl = tiles_x * nrows tiles (MCU rows my0 ..), then the tiles
// its tickets name (`ticket`: zeroed, one per launch). Quantiser tables, histogram and mbarrier are set up once per
// CTA, the histogram is flushed once. While a tile is coded, the bulk copies of the CTA's next tile land in the staged-row region at the end of the token area.
template <int HS, int VS, bool DUMP, int NC = 3>
__global__ void __launch_bounds__(256, 3)
k_fdct(const uint8_t *__restrict__ img, size_t step, Geom g, const QuantDev *__restrict__ qd,
       uint32_t *__restrict__ pool, uint32_t *__restrict__ pool_count, uint32_t *__restrict__ ticket, TileRec *__restrict__ recs,
       uint32_t *__restrict__ ghist, int do_hist, int bulk_ok, int my0, int nrows, int16_t *__restrict__ coef) {
    using C = K1<HS, VS, NC>;
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t *raw = smem + C::OFF_RAW;
    uint32_t *tok = reinterpret_cast<uint32_t *>(smem);
    uint8_t *Yp = smem + C::OFF_Y, *Cbp = smem + C::OFF_CB, *Crp = smem + C::OFF_CR;
    float *qs = reinterpret_cast<float *>(smem + C::OFF_Q);
    uint32_t *hs = reinterpret_cast<uint32_t *>(smem + C::OFF_HIST);
    int16_t *dcs = reinterpret_cast<int16_t *>(smem + C::OFF_DC);
    uint32_t *misc = reinterpret_cast<uint32_t *>(smem + C::OFF_MISC);
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem + C::OFF_BAR);

    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int ntl = g.tiles_x * nrows;

    // once per CTA: quantisation constants, histogram, mbarrier; then the first tile's rows are requested
    if (tid < 128) qs[tid] = qd->finv[tid >> 6][tid & 63];
    else if (tid < 192) qs[tid] = 0.0f;   // reciprocal 0: every coefficient of a dummy block quantises to 0
    if (do_hist)
        for (int i = tid; i < 1024; i += 256) hs[i] = 0;
    if (tid == 0) {
        mbar_init(bar, 1);
        mbar_fence_init();
    }
    __syncthreads();
    if (bulk_ok && tid == 0) stage_rows<HS, VS, NC>(img, step, g, my0, blockIdx.x, ntl, raw, bar);

    // Stage B needs all 80 registers, so nothing of the loop may stay live through it: the tile index and the mbarrier
    // parity are parked in shared memory (misc[11], misc[12]; misc[13]: the tile's first block for DUMP; misc[14]: the
    // next tile), written by
    // thread 0 before the barrier that ends stage A and read back with volatile loads after stage B. (For the same
    // reason stage B sets xin[] for idle threads too.)
    int t = blockIdx.x;
    uint32_t phase = 0;   // parity of the mbarrier phase the next staged tile completes
    while (t < ntl) {
        const TilePos P = tile_pos<C::MCU_W, C::MCU_H>(g, my0, t);
        const int my = P.my, mx0 = P.mx0, nmcu = P.nmcu, x0 = P.x0, y0 = P.y0, tile_px = P.tile_px;
        const int nblk = nmcu * C::BPM;

        if (P.interior) {
            if (bulk_ok) {
                mbar_wait(bar, phase);
                phase ^= 1u;
            } else {
                const unsigned row_bytes = (unsigned)tile_px * NC;
                const uint8_t *src = img + (size_t)y0 * step + (size_t)x0 * NC;
                for (int r = 0; r < C::MCU_H; r++)
                    for (int i = tid; i < (int)row_bytes; i += 256) raw[r * C::RAW_STRIDE + i] = src[(size_t)r * step + i];
                __syncthreads();
            }
            // ---- stage A (fast): one warp per row group (VS pixel rows), 8 pixels per lane and step (gray: nothing to do)
            const int ngx = NC == 1 ? 0 : nmcu * HS;
            const int rg = wid;
            for (int gx = lane; gx < ngx; gx += 32) {
                // jccolor.c rgb_ycc_convert on packed pixels: every component is two 2-way dot products (IDP.2A, 16-bit
                // coefficients x the pixel's bytes [b, g | r, next b]); for the chroma planes t = (N + 32768) >> 16 with
                // N = -(the libjpeg sum without its constant), so that cb = 128 - t exactly (floor identities).
                int tbv[VS][8], trv[VS][8];
#pragma unroll
                for (int v = 0; v < VS; v++) {
                    const int r = rg * VS + v;
                    const uint2 *p = reinterpret_cast<const uint2 *>(raw + r * C::RAW_STRIDE + gx * 24);
                    const uint2 a = p[0], b = p[1], c = p[2];
                    const uint32_t w[6] = {a.x, a.y, b.x, b.y, c.x, c.y};
                    uint32_t S[8];
#pragma unroll
                    for (int px = 0; px < 8; px++) {
                        const int o = 3 * px, wi = o >> 2, bo = o & 3;
                        // bytes [b, g, r, *] of pixel px (the fourth byte meets a zero coefficient)
                        const uint32_t q = bo == 0 ? w[wi] : (bo == 1 ? (w[wi] >> 8) : __byte_perm(w[wi], w[wi + 1], bo == 2 ? 0x5432 : 0x6543));
                        S[px] = dp2a_hi_uu(B2J_PAIR(19595, 0), q, dp2a_lo_uu(B2J_PAIR(7471, 38470), q, 32768u));
                        tbv[v][px] = dp2a_hi_su(B2J_PAIR(11059, 0), q, dp2a_lo_su(B2J_PAIR(-32768, 21709), q, 32768)) >> 16;
                        trv[v][px] = dp2a_hi_su(B2J_PAIR(-32768, 0), q, dp2a_lo_su(B2J_PAIR(5329, 27439), q, 32768)) >> 16;
                    }
                    // y = S >> 16 (S < 2^24): byte 2 of every sum
                    const uint32_t y0 = __byte_perm(__byte_perm(S[0], S[1], 0x0062), __byte_perm(S[2], S[3], 0x0062), 0x5410);
                    const uint32_t y1 = __byte_perm(__byte_perm(S[4], S[5], 0x0062), __byte_perm(S[6], S[7], 0x0062), 0x5410);
                    *reinterpret_cast<uint2 *>(Yp + r * C::Y_STRIDE + gx * 8) = make_uint2(y0, y1);
                }
                // jcsample.c: fullsize / h2v1 (bias 0,1) / h2v2 (bias 1,2) / int_downsample (h1v2, h4v1), with cb = 128 - t
                uint32_t ob[2] = {0, 0}, orr[2] = {0, 0};
#pragma unroll
                for (int j = 0; j < 8 / HS; j++) {
                    int sb = 0, sr = 0;
#pragma unroll
                    for (int v = 0; v < VS; v++)
#pragma unroll
                        for (int h = 0; h < HS; h++) {
                            sb += tbv[v][j * HS + h];
                            sr += trv[v][j * HS + h];
                        }
                    constexpr int K = 128 * HS * VS;
                    int ocb, ocr;
                    if (HS == 1 && VS == 1) { ocb = K - sb; ocr = K - sr; }
                    else if (HS == 2 && VS == 1) { ocb = (K + (j & 1) - sb) >> 1; ocr = (K + (j & 1) - sr) >> 1; }
                    else if (HS == 2 && VS == 2) { ocb = (K + 1 + (j & 1) - sb) >> 2; ocr = (K + 1 + (j & 1) - sr) >> 2; }
                    else if (HS == 1 && VS == 2) { ocb = (K + 1 - sb) >> 1; ocr = (K + 1 - sr) >> 1; }
                    else { ocb = (K + 2 - sb) >> 2; ocr = (K + 2 - sr) >> 2; }
                    ob[j >> 2] |= (uint32_t)ocb << ((j & 3) * 8);
                    orr[j >> 2] |= (uint32_t)ocr << ((j & 3) * 8);
                }
                uint8_t *dcb = Cbp + rg * C::C_STRIDE + gx * (8 / HS), *dcr = Crp + rg * C::C_STRIDE + gx * (8 / HS);
                if (HS == 1) {
                    *reinterpret_cast<uint2 *>(dcb) = make_uint2(ob[0], ob[1]);
                    *reinterpret_cast<uint2 *>(dcr) = make_uint2(orr[0], orr[1]);
                } else if (HS == 2) {
                    *reinterpret_cast<uint32_t *>(dcb) = ob[0];
                    *reinterpret_cast<uint32_t *>(dcr) = orr[0];
                } else {
                    *reinterpret_cast<uint16_t *>(dcb) = (uint16_t)ob[0];
                    *reinterpret_cast<uint16_t *>(dcr) = (uint16_t)orr[0];
                }
            }
        } else if (NC == 1) {
            // ---- edge tiles, gray: the last column / row replicated (jcsample.c expand_right_edge, jcprepct.c)
            for (int i = tid; i < C::MCU_H * tile_px; i += 256) {
                const int r = i / tile_px, x = i - r * tile_px;
                const int yy = min(y0 + r, g.H - 1), xx = min(x0 + x, g.W - 1);
                Yp[r * C::Y_STRIDE + x] = img[(size_t)yy * step + (size_t)xx];
            }
        } else {
            // ---- stage A (edge tiles): per-sample with libjpeg's padding rules (jcprepct.c / jcsample.c expand_right_edge)
            for (int i = tid; i < C::MCU_H * tile_px; i += 256) {
                const int r = i / tile_px, x = i - r * tile_px;
                const int yy = min(y0 + r, g.H - 1), xx = min(x0 + x, g.W - 1);
                const uint8_t *p = img + (size_t)yy * step + (size_t)xx * 3;
                int y, cb, cr;
                ycc(p[0], p[1], p[2], y, cb, cr);
                Yp[r * C::Y_STRIDE + x] = (uint8_t)y;
            }
            const int cw = nmcu * 8;
            for (int i = tid; i < 8 * cw; i += 256) {
                const int rd = i / cw, j = i - rd * cw;
                const int rs = min(my * 8 + rd, g.dh[1] - 1);  // replicate the last DOWNSAMPLED row
                const int jg = mx0 * 8 + j;
                int sb = 0, sr = 0;
                for (int v = 0; v < VS; v++) {
                    const int yy = min(rs * VS + v, g.H - 1);   // replicate the last pixel row
                    for (int h = 0; h < HS; h++) {
                        const int xx = min(jg * HS + h, g.W - 1);
                        const uint8_t *p = img + (size_t)yy * step + (size_t)xx * 3;
                        int y, cb, cr;
                        ycc(p[0], p[1], p[2], y, cb, cr);
                        sb += cb;
                        sr += cr;
                    }
                }
                int ocb, ocr;
                if (HS == 1 && VS == 1) { ocb = sb; ocr = sr; }
                else if (HS == 2 && VS == 1) { ocb = (sb + (jg & 1)) >> 1; ocr = (sr + (jg & 1)) >> 1; }
                else if (HS == 2 && VS == 2) { ocb = (sb + 1 + (jg & 1)) >> 2; ocr = (sr + 1 + (jg & 1)) >> 2; }
                else if (HS == 1 && VS == 2) { ocb = (sb + 1) >> 1; ocr = (sr + 1) >> 1; }
                else { ocb = (sb + 2) >> 2; ocr = (sr + 2) >> 2; }
                Cbp[rd * C::C_STRIDE + j] = (uint8_t)ocb;
                Crp[rd * C::C_STRIDE + j] = (uint8_t)ocr;
            }
        }
        if (tid == 0) { misc[11] = (uint32_t)t; misc[12] = phase; misc[13] = (uint32_t)((my * g.mcux + mx0) * C::BPM); }
        __syncthreads();  // planes complete; raw is dead, the token area may be written

        // ---- stage B: one thread per block
        const int blk = tid;
        const bool active = blk < nblk;
        const int m = blk / C::BPM, bn = blk - m * C::BPM;
        const bool isY = bn < C::HV;
        const int by = isY ? bn / HS : 0, bx = isY ? bn - by * HS : 0;
        const int tbl = isY ? 0 : 1;
        const int comp = isY ? 0 : bn - C::HV + 1;
        bool real = true;
        if (isY) real = ((mx0 + m) * HS + bx < g.wib[0]) && (my * VS + by < g.hib[0]);
        int ntok = 0;
        int mydc = 0;
        uint32_t pk[32];   // quantised coefficients, zig-zag order, two per word
        int v[64];
        uint32_t xin[16] = {};   // the block's samples, one row per word pair (set for idle threads too: inside
                                 // the tile loop an unset array would carry the previous tile's values)
        if (active) {
            const uint8_t *src;
            int stride;
            if (isY) { src = Yp + (by * 8) * C::Y_STRIDE + (m * HS + bx) * 8; stride = C::Y_STRIDE; }
            else { src = (bn == C::HV ? Cbp : Crp) + m * 8; stride = C::C_STRIDE; }
#pragma unroll
            for (int r = 0; r < 8; r++) {
                const uint2 w = *reinterpret_cast<const uint2 *>(src + r * stride);
                xin[2 * r] = w.x;       // level shift folded into the DC term below
                xin[2 * r + 1] = w.y;
            }
        }
        __syncthreads();  // every sample is in registers: the planes are dead, the token area may be written
        if (active) {
            fdct_rows_k<0>(xin, v); fdct_rows_k<1>(xin, v); fdct_rows_k<2>(xin, v); fdct_rows_k<3>(xin, v);
            fdct_rows_k<4>(xin, v); fdct_rows_k<5>(xin, v); fdct_rows_k<6>(xin, v); fdct_rows_k<7>(xin, v);
#pragma unroll
            for (int c = 0; c < 8; c++)
                fdct8<true>(v[c], v[8 + c], v[16 + c], v[24 + c], v[32 + c], v[40 + c], v[48 + c], v[56 + c]);
            v[0] -= 8192;  // 64 samples x 128: the only output the -128 level shift changes (exact: multiple of 4)

            // quantise (jcdctmgr.c): q = sign(c) * ((|c| + d/2) / d), d = 8*qtbl, on the FMA pipes, which the integer
            // transform leaves idle. The table holds finv = fl32((1 + 2^-20) / d) * 4096: the single rounding of
            // fma(c, finv, 1.5 * 2^35) lands on 4096 * that quotient for every divisor and |c| <= 2^18 (ties of |c|/d go away
            // from zero because finv is a little large, everything else is further than |c| * 2^-20 from a tie), i.e. the
            // quotient is the low half of the result's bit pattern. The same table value counts the non-zero AC
            // coefficients (one token each) with ONE saturating FMA: |c| * finv - 2047 is >= 1 from |c| = d/2 on and
            // negative below. Both checked exhaustively on the CPU (tests/cpp/quant_exhaustive.c). Results are kept as
            // 16-bit pairs in zig-zag order (they live across the CTA scan below).
            const float4 *qt = reinterpret_cast<const float4 *>(qs + ((C::HV > 1 && !real) ? 2 : tbl) * 64);
            constexpr float MAGIC = 12582912.0f;        // 1.5 * 2^23: int -> float
            constexpr float MAGICK = 51539607552.0f;    // 1.5 * 2^35: bit pattern 0x51400000 + quotient
            float nnzf = 0.0f;
#pragma unroll
            for (int n4 = 0; n4 < 16; n4++) {
                const float4 qv = qt[n4];
                const float qq[4] = {qv.x, qv.y, qv.z, qv.w};
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    const int n = n4 * 4 + j;
                    const float xf = __int_as_float(v[n] + 0x4B400000) - MAGIC;   // exact int -> float for |c| < 2^22
                    if (n != 0) nnzf += __saturatef(fmaf(fabsf(xf), qq[j], -2047.0f));
                    v[n] = __float_as_int(fmaf(xf, qq[j], MAGICK));
                }
            }
            mydc = v[0] - 0x51400000;
#pragma unroll
            for (int k = 0; k < 64; k += 2) pk[k >> 1] = __byte_perm((uint32_t)v[zigzag_nat(k)], (uint32_t)v[zigzag_nat(k + 1)], 0x5410);
            ntok = 1 + (int)nnzf + ((pk[31] >> 16) == 0u ? 1 : 0);   // DC, one per non-zero AC, EOB iff the last coefficient is zero
            if constexpr (DUMP) {   // quantised coefficients, scan order, zig-zag inside the block
                uint4 *cdst = reinterpret_cast<uint4 *>(coef + ((size_t)ld_volatile_shared(misc + 13) + blk) * 64);
                if (real || C::HV == 1) {
#pragma unroll
                    for (int c = 0; c < 8; c++) cdst[c] = make_uint4(pk[4 * c], pk[4 * c + 1], pk[4 * c + 2], pk[4 * c + 3]);
                }
            }
            if (real) dcs[blk] = (int16_t)mydc;
        }
        __syncthreads();

        // ---- dummy blocks (jccoefct.c compress_data): zero AC, DC of the last real block before them in the MCU
        if (C::HV > 1) {
            const TilePos D = tile_pos<C::MCU_W, C::MCU_H>(g, my0, (int)ld_volatile_shared(misc + 11));
            if (active && !real) {
                const int nrx = min(HS, g.wib[0] - (D.mx0 + m) * HS), nry = min(VS, g.hib[0] - D.my * VS);
                const int sby = min(by, nry - 1);
                const int sblk = m * C::BPM + sby * HS + (nrx - 1);
                mydc = dcs[sblk];
            }
            __syncthreads();
            if (active && !real) {
                dcs[blk] = (int16_t)mydc;
                if constexpr (DUMP) {
                    uint4 *cdst = reinterpret_cast<uint4 *>(coef + ((size_t)ld_volatile_shared(misc + 13) + blk) * 64);
#pragma unroll
                    for (int c = 0; c < 8; c++) cdst[c] = make_uint4(c == 0 ? ((uint32_t)mydc & 0xFFFFu) : 0u, 0u, 0u, 0u);
                }
            }
            __syncthreads();
        }

        // ---- DC token: difference to the previous block of the same component; predecessors outside the tile are
        //      resolved later by k_dc_edge_hist from TileRec.last_dc (the token carries the raw DC until then)
        uint32_t t0 = 0;
        if (active) {
            int pb = -1;
            if (isY) pb = bn > 0 ? blk - 1 : (m > 0 ? blk - C::BPM + C::HV - 1 : -1);
            else pb = m > 0 ? blk - C::BPM : -1;
            if (pb >= 0) t0 = ((uint32_t)(2 + tbl) << 16) | ((uint32_t)(mydc - (int)dcs[pb]) & 0xFFFFu);   // stage C sizes it
            else t0 = TOK_RAWDC | ((uint32_t)(2 + tbl) << 16) | ((uint32_t)comp << 18) | ((uint32_t)mydc & 0xFFFFu);
        }

        // ---- place of every block in the tile's token run: CTA scan of the token counts
        uint32_t inc = (uint32_t)ntok;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += y;
        }
        if (lane == 31) misc[wid] = inc;
        __syncthreads();
        uint32_t off = inc - (uint32_t)ntok, total = 0;
#pragma unroll
        for (int w = 0; w < 8; w++) { const uint32_t x = misc[w]; if (w < wid) off += x; total += x; }
        if (NC == 3 && tid == C::HV) misc[9] = off;        // run offsets of the first MCU's chroma DC tokens
        if (NC == 3 && tid == C::HV + 1) misc[10] = off;

        // ---- run-length walk (jchuff.c encode_one_block): one entry per non-zero AC coefficient, straight to its slot:
        //      the token's run / ZRL-count and table fields | coefficient: the run counter advances by TOK_RUN_STEP, which
        //      puts the run where the token wants it and adds it to the table field (common.cuh). The divergent region is the
        //      store and the reset of the run counter; sizes and value bits are derived in stage C with full warps.
        if (active) {
            uint32_t sa = smem_u32(tok + off);
            asm volatile("st.shared.u32 [%0], %1;" ::"r"(sa), "r"(t0) : "memory");
            sa += 4;
            const uint32_t rbase = (uint32_t)tbl << 16;   // tcode of the block's AC table
            uint32_t r = rbase;
#pragma unroll
            for (int k = 1; k < 64; k++) {
                const uint32_t p2 = pk[k >> 1];
                const bool nzk = (k & 1) ? (p2 >= 0x10000u) : ((p2 & 0xFFFFu) != 0u);
                if (nzk) {
                    const uint32_t e = (k & 1) ? __byte_perm(p2, r, 0x7632) : ((p2 & 0xFFFFu) | r);
                    asm volatile("st.shared.u32 [%0], %1;" ::"r"(sa), "r"(e) : "memory");
                    sa += 4;
                    r = rbase - TOK_RUN_STEP;
                }
                r += TOK_RUN_STEP;
            }
            if (pk[31] < 0x10000u) asm volatile("st.shared.u32 [%0], %1;" ::"r"(sa), "r"(rbase) : "memory");   // EOB
        }
        __syncthreads();
        t = (int)ld_volatile_shared(misc + 11);   // the tile's index and the parity come back
        phase = ld_volatile_shared(misc + 12);
        if (tid == 0) {
            const int nlast = tile_pos<C::MCU_W, C::MCU_H>(g, my0, t).nmcu * C::BPM;
            // the CTA's next tile comes from the launch's ticket (tiles 0 .. gridDim.x - 1 are the first ones): tiles
            // differ in cost (remainder tiles, token counts), so a fixed order would leave some CTAs a longer tail
            const uint32_t nt = gridDim.x + atomicAdd(ticket, 1u);
            const uint32_t base = atomicAdd(pool_count, total);
            misc[8] = base;
            misc[14] = nt;
            TileRec r;
            r.base = base; r.count = total;
            if (NC == 1) {
                r.pos_cb = r.pos_cr = 0;
                r.first_dc[0] = dcs[0]; r.first_dc[1] = r.first_dc[2] = 0;
                r.last_dc[0] = dcs[nlast - 1]; r.last_dc[1] = r.last_dc[2] = 0;
            } else {
                r.pos_cb = (uint16_t)misc[9]; r.pos_cr = (uint16_t)misc[10];
                r.first_dc[0] = dcs[0]; r.first_dc[1] = dcs[C::HV]; r.first_dc[2] = dcs[C::HV + 1];
                r.last_dc[0] = dcs[nlast - 3]; r.last_dc[1] = dcs[nlast - 2]; r.last_dc[2] = dcs[nlast - 1];
            }
            recs[my0 * g.tiles_x + t] = r;
        }
        __syncthreads();
        t = (int)misc[14];
        // a run that leaves the staged-row region alone lets the next tile's rows land while this one is coded
        const bool early = total <= (uint32_t)C::OFF_RAW / 4u;
        if (early && bulk_ok && tid == 0) stage_rows<HS, VS, NC>(img, step, g, my0, t, ntl, raw, bar);

        // ---- stage C: the run in output order -> final tokens, symbol statistics, coalesced stores
        if (do_hist) stage_c<true, NC>(tok, pool + (size_t)misc[8], total, hs, tid);
        else stage_c<false, NC>(tok, pool + (size_t)misc[8], total, hs, tid);
        __syncthreads();   // the run is read: the next tile may write planes and staged rows over it
        if (!early && bulk_ok && tid == 0) stage_rows<HS, VS, NC>(img, step, g, my0, t, ntl, raw, bar);
    }

    if (do_hist) {   // the CTA's symbol counts, once: token bins (common.cuh) -> (table, symbol)
        for (int i = tid; i < 1024; i += 256) {
            const uint32_t n = hs[i];
            if (n) atomicAdd(&ghist[bin_table(i) * 257 + bin_symbol(i)], n);
        }
    }
}

// DC-difference symbols of each fdct tile's first MCU (their predecessor block lives in the previous tile; the
// strip's very first MCU takes pred_in), plus the strip's last DCs for the next strip. With `resolve` the three
// raw-DC tokens of every tile are rewritten in the pool as final difference tokens, so the entropy coder sees one
// uniform token format. With `xr` (one-collective strip exchange) the strip's first MCU is left alone -- its
// predictors arrive with the exchange, k_strip_merge finishes it -- and the record's DC / first-token fields are filled.
// NC: DCs per tile edge (components per image; gray has one raw-DC token per tile).
template <int NC>
__global__ void __launch_bounds__(256)
k_dc_edge_hist(const TileRec *__restrict__ recs, Geom g, const int16_t *__restrict__ pred_in,
               uint32_t *__restrict__ ghist, int16_t *__restrict__ last_dc, int do_hist,
               uint32_t *__restrict__ pool, int resolve, StripRecord *__restrict__ xr, int rst_tiles) {
    __shared__ uint32_t s_h[2][16];   // DC categories 0..11 of the two DC tables, aggregated per CTA
    pdl_trigger();
    pdl_wait();
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int ntile = g.tiles_x * g.mcuy;
    if (threadIdx.x < 32) s_h[threadIdx.x >> 4][threadIdx.x & 15] = 0;
    __syncthreads();
    if (t < ntile * NC && (do_hist || resolve) && !(xr && t < NC)) {
        const int tile = t / NC, c = t - tile * NC;
        const TileRec r = recs[tile];
        const int dc = r.first_dc[c];
        // restart intervals (rst_tiles = tiles per interval, whole MCU rows): predictors return to 0 at an interval start
        const int pd = tile == 0 ? pred_in[c] : ((rst_tiles && tile % rst_tiles == 0) ? 0 : recs[tile - 1].last_dc[c]);
        const int diff = dc - pd;
        const int nb = nbits_of(diff);
        if (do_hist) atomicAdd(&s_h[c ? 1 : 0][nb & 15], 1u);
        if (resolve) {
            const uint32_t p = c == 0 ? 0u : (c == 1 ? r.pos_cb : r.pos_cr);
            pool[r.base + p] = tok_dc(c ? 2u : 0u, (uint32_t)nb, (uint32_t)(diff + (diff >> 31)) & ((1u << nb) - 1u));
        }
    }
    if (t < NC) last_dc[t] = recs[ntile - 1].last_dc[t];
    if (xr) {
        if (t < NC) xr->first_dc[t] = recs[0].first_dc[t];
        if (t >= 32 && t < 40) {   // tile 0 only: the other tiles' first tokens are being rewritten by this launch
            const uint32_t n = min(recs[0].count, 8u), j = (uint32_t)t - 32u;
            xr->tok[j] = j < n ? pool[recs[0].base + j] : 0u;
            if (j == 0) xr->ntok = n;
        }
    }
    __syncthreads();
    if (do_hist && threadIdx.x < 32) {
        const uint32_t n = s_h[threadIdx.x >> 4][threadIdx.x & 15];
        if (n) atomicAdd(&ghist[(threadIdx.x >> 4) * 2 * 257 + (threadIdx.x & 15)], n);
    }
}

template <int HS, int VS, bool DUMP, int NC>
static cudaError_t launch_one2(const uint8_t *img, size_t step, const Geom &g, const QuantDev *qd, uint32_t *pool,
                               uint32_t *pool_count, uint32_t *ticket, TileRec *recs, uint32_t *hist, int do_hist, int my0, int nrows,
                               int16_t *coef, cudaStream_t s) {
    using C = K1<HS, VS, NC>;
    constexpr int SM = C::SMEM;
    // the attribute is per device: one bit per device ordinal (a process may hold contexts on several GPUs)
    static std::atomic<uint64_t> attr_done{0};
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    const uint64_t bit = 1ull << (dev & 63);
    if (!(attr_done.load(std::memory_order_acquire) & bit)) {
        e = cudaFuncSetAttribute(k_fdct<HS, VS, DUMP, NC>, cudaFuncAttributeMaxDynamicSharedMemorySize, SM);
        if (e != cudaSuccess) return e;
        attr_done.fetch_or(bit, std::memory_order_release);
    }
    // TMA bulk copies need 16-byte aligned global addresses and sizes for every row of every interior tile
    const int row_unit = g.tm * C::MCU_W * NC;  // byte offset between tiles in a row
    int bulk_ok = ((reinterpret_cast<uintptr_t>(img) & 15) == 0) && (step % 16 == 0) && (row_unit % 16 == 0);
    // the last tile of a row may hold fewer MCUs: its byte count must be a multiple of 16 as well
    const int last_n = g.mcux - (g.tiles_x - 1) * g.tm;
    if ((last_n * C::MCU_W * NC) % 16 != 0 && (long long)g.mcux * C::MCU_W <= g.W) bulk_ok = 0;
    // persistent CTAs: as many as are resident at once (three per SM), never more than there are tiles
    int nsm = 0;
    e = cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess) return e;
    const int ntl = g.tiles_x * nrows;
    if (ntl <= 0) return cudaSuccess;
    const int grid = std::min(ntl, 3 * nsm);
    k_fdct<HS, VS, DUMP, NC><<<grid, 256, SM, s>>>(img, step, g, qd, pool, pool_count, ticket, recs, hist, do_hist, bulk_ok, my0, nrows, coef);
    return cudaGetLastError();
}

template <int HS, int VS, int NC = 3>
static cudaError_t launch_one(const uint8_t *img, size_t step, const Geom &g, const QuantDev *qd, uint32_t *pool,
                              uint32_t *pool_count, uint32_t *ticket, TileRec *recs, uint32_t *hist, int do_hist, int my0, int nrows,
                              int16_t *coef, cudaStream_t s) {
    return coef ? launch_one2<HS, VS, true, NC>(img, step, g, qd, pool, pool_count, ticket, recs, hist, do_hist, my0, nrows, coef, s)
                : launch_one2<HS, VS, false, NC>(img, step, g, qd, pool, pool_count, ticket, recs, hist, do_hist, my0, nrows, coef, s);
}

int fdct_tm_max(int hs, int vs, int nc) { return (256 / (nc == 1 ? 1 : hs * vs + 2)) & ~1; }

cudaError_t launch_fdct(const uint8_t *img, size_t step, const Geom &g, const QuantDev *qd, uint32_t *pool,
                        uint32_t *pool_count, uint32_t *ticket, TileRec *recs, uint32_t *hist, int do_hist, int my0, int nrows,
                        int16_t *coef_dump, cudaStream_t s) {
#define B2J_ARGS img, step, g, qd, pool, pool_count, ticket, recs, hist, do_hist, my0, nrows, coef_dump, s
    if (g.nc == 1) return launch_one<1, 1, 1>(B2J_ARGS);
    if (g.hs == 1 && g.vs == 1) return launch_one<1, 1>(B2J_ARGS);
    if (g.hs == 2 && g.vs == 1) return launch_one<2, 1>(B2J_ARGS);
    if (g.hs == 1 && g.vs == 2) return launch_one<1, 2>(B2J_ARGS);
    if (g.hs == 2 && g.vs == 2) return launch_one<2, 2>(B2J_ARGS);
    if (g.hs == 4 && g.vs == 1) return launch_one<4, 1>(B2J_ARGS);
#undef B2J_ARGS
    return cudaErrorInvalidValue;
}

cudaError_t launch_dc_edge_hist(const TileRec *recs, const Geom &g, const int16_t *pred_in, uint32_t *hist,
                                int16_t *last_dc, int do_hist, uint32_t *pool, int resolve, StripRecord *xr, int rst_tiles, cudaStream_t s) {
    const int n = max(64, g.tiles_x * g.mcuy * g.nc);
    if (g.nc == 1)
        return launch_pdl(k_dc_edge_hist<1>, dim3((n + 255) / 256), dim3(256), 0, s, recs, g, pred_in, hist, last_dc, do_hist, pool, resolve, xr, rst_tiles);
    return launch_pdl(k_dc_edge_hist<3>, dim3((n + 255) / 256), dim3(256), 0, s, recs, g, pred_in, hist, last_dc, do_hist, pool, resolve, xr, rst_tiles);
}

}  // namespace b2j
