/*
 * jpeg_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE (see jpeg_oracle.h).
 *
 * Plain-C restatement of libjpeg-turbo 3.1.2 baseline JPEG (DCT_ISLOW, fancy upsampling; restart intervals
 * in orc_encode_rst / the decoder; progressive mode in orc_encode_progressive / the decoder; one-component files;
 * gray and reduced-size output) following SURVEY.md Appendix A section by section. The reference repository contains no
 * JPEG arithmetic of its own (it calls nvjpegEncodeImage at ImageCompressorImpl.cu:280 and the
 * nvjpegDecodeJpeg* trio at :364-366); the north-star pins results to libjpeg-turbo instead.
 * Pinned by tests/test_oracle_golden.py (live cv2 = libjpeg-turbo 3.1.2) and tests/golden/.
 */
#include "jpeg_oracle.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>

/* ------------------------------------------------------------------ tables */

static const uint8_t ZIGZAG[64] = { /* zig-zag index -> natural index (jutils.c jpeg_natural_order) */
    0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
    41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
    30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};

static const uint8_t BASE_LUMA[64] = { /* jcparam.c std_luminance_quant_tbl (Annex K.1) */
    16, 11, 10, 16, 24,  40,  51,  61,  12, 12, 14, 19, 26,  58,  60,  55,
    14, 13, 16, 24, 40,  57,  69,  56,  14, 17, 22, 29, 51,  87,  80,  62,
    18, 22, 37, 56, 68,  109, 103, 77,  24, 35, 55, 64, 81,  104, 113, 92,
    49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99};

static const uint8_t BASE_CHROMA[64] = { /* jcparam.c std_chrominance_quant_tbl (Annex K.2) */
    17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99, 24, 26, 56, 99, 99, 99,
    99, 99, 47, 66, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99,
    99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99};

/* Annex K.3-K.6 (jcparam.c std_huff_tables) */
static const uint8_t STD_DC_LUMA_BITS[17] = {0, 0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0};
static const uint8_t STD_DC_CHROMA_BITS[17] = {0, 0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0};
static const uint8_t STD_DC_VAL[12] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11};
static const uint8_t STD_AC_LUMA_BITS[17] = {0, 0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 0x7d};
static const uint8_t STD_AC_LUMA_VAL[162] = {
    0x01, 0x02, 0x03, 0x00, 0x04, 0x11, 0x05, 0x12, 0x21, 0x31, 0x41, 0x06, 0x13, 0x51, 0x61, 0x07, 0x22, 0x71,
    0x14, 0x32, 0x81, 0x91, 0xa1, 0x08, 0x23, 0x42, 0xb1, 0xc1, 0x15, 0x52, 0xd1, 0xf0, 0x24, 0x33, 0x62, 0x72,
    0x82, 0x09, 0x0a, 0x16, 0x17, 0x18, 0x19, 0x1a, 0x25, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x34, 0x35, 0x36, 0x37,
    0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59,
    0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a, 0x83,
    0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a, 0xa2, 0xa3,
    0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3,
    0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe1, 0xe2,
    0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf1, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa};
static const uint8_t STD_AC_CHROMA_BITS[17] = {0, 0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 0x77};
static const uint8_t STD_AC_CHROMA_VAL[162] = {
    0x00, 0x01, 0x02, 0x03, 0x11, 0x04, 0x05, 0x21, 0x31, 0x06, 0x12, 0x41, 0x51, 0x07, 0x61, 0x71, 0x13, 0x22,
    0x32, 0x81, 0x08, 0x14, 0x42, 0x91, 0xa1, 0xb1, 0xc1, 0x09, 0x23, 0x33, 0x52, 0xf0, 0x15, 0x62, 0x72, 0xd1,
    0x0a, 0x16, 0x24, 0x34, 0xe1, 0x25, 0xf1, 0x17, 0x18, 0x19, 0x1a, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x35, 0x36,
    0x37, 0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58,
    0x59, 0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a,
    0x82, 0x83, 0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a,
    0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba,
    0xc2, 0xc3, 0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda,
    0xe2, 0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa};

static int ceil_div(int a, int b) { return (a + b - 1) / b; }
static int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

/* ------------------------------------------------------------------ geometry (jcmaster.c initial_setup / per_scan_setup) */

static const int HS[5] = {1, 2, 1, 2, 4}, VS[5] = {1, 1, 2, 2, 1};

static int css_of(int hs, int vs) {
    for (int i = 0; i < 5; i++) if (HS[i] == hs && VS[i] == vs) return i;
    return -1;
}

/* css 0..4: three components, chroma 1x1; ORC_CSS_GRAY: one component, one block per MCU (a one-component scan is
 * non-interleaved, so its sampling factors do not matter) */
static void layout(int W, int H, int css, orc_geom *g) {
    const int nc = css == ORC_CSS_GRAY ? 1 : 3;
    memset(g, 0, sizeof(*g));
    g->W = W; g->H = H; g->css = css;
    g->hs = nc == 1 ? 1 : HS[css]; g->vs = nc == 1 ? 1 : VS[css];
    g->mcux = ceil_div(W, 8 * g->hs);
    g->mcuy = ceil_div(H, 8 * g->vs);
    g->bpm = nc == 1 ? 1 : g->hs * g->vs + 2;
    for (int c = 0; c < nc; c++) {
        int h = c ? 1 : g->hs, v = c ? 1 : g->vs;
        g->dw[c] = ceil_div(W * h, g->hs);
        g->dh[c] = ceil_div(H * v, g->vs);
        g->wib[c] = ceil_div(g->dw[c], 8);
        g->hib[c] = ceil_div(g->dh[c], 8);
    }
    g->nblocks = (long long)g->mcux * g->mcuy * g->bpm;
}

int orc_geometry(int W, int H, int css, orc_geom *g) {
    if (W <= 0 || H <= 0 || css < 0 || css > 4) return -1;
    layout(W, H, css, g);
    return 0;
}

/* ------------------------------------------------------------------ A.1 quant tables (jcparam.c jpeg_quality_scaling / jpeg_add_quant_table) */

void orc_quant_tables(int quality, uint16_t qt[2][64]) {
    int q = clampi(quality, 1, 100);
    int scale = q < 50 ? 5000 / q : 200 - 2 * q;
    for (int i = 0; i < 64; i++) {
        long a = ((long)BASE_LUMA[i] * scale + 50) / 100;
        long b = ((long)BASE_CHROMA[i] * scale + 50) / 100;
        qt[0][i] = (uint16_t)clampi((int)a, 1, 255); /* force_baseline */
        qt[1][i] = (uint16_t)clampi((int)b, 1, 255);
    }
}

/* ------------------------------------------------------------------ Appendix B generator */

static uint32_t hash32(uint32_t x, uint32_t y, uint32_t c, uint32_t s) {
    uint32_t h = x * 0x9E3779B1u ^ y * 0x85EBCA77u ^ c * 0xC2B2AE3Du ^ s * 0x27D4EB2Fu;
    h ^= h >> 15; h *= 0x2C1B3C6Du; h ^= h >> 12; h *= 0x297A2D39u; h ^= h >> 15;
    return h;
}
static int fmod_i(long long v, int m) { long long r = v % m; return (int)(r < 0 ? r + m : r); }
static int tri(long long v, int P) { int t = fmod_i(v, 2 * P) - P; if (t < 0) t = -t; return t * 255 / P; }

void orc_synth_rows(int W, int H, int y0, int rows, uint32_t seed, int amp, uint8_t *out) {
    (void)H;
    for (int yy = 0; yy < rows; yy++) {
        int y = y0 + yy;
        for (int x = 0; x < W; x++) {
            int cell = (int)(hash32((uint32_t)(x >> 5), (uint32_t)(y >> 5), 7, seed) & 63) - 32;
            for (int c = 0; c < 3; c++) {
                int base = (tri((long long)x + 3LL * y + 37 * c, 512) + tri(5LL * x - 2LL * y + 91 * c, 160) +
                            tri((long long)y + 11 * c, 2048)) / 3;
                int noise = (int)(hash32((uint32_t)x, (uint32_t)y, (uint32_t)c, seed) % (uint32_t)(2 * amp + 1)) - amp;
                out[((size_t)yy * W + x) * 3 + c] = (uint8_t)clampi(base + cell + noise, 0, 255);
            }
        }
    }
}
void orc_synth(int W, int H, uint32_t seed, int amp, uint8_t *out) { orc_synth_rows(W, H, 0, H, seed, amp, out); }

/* ------------------------------------------------------------------ A.2 colour (jccolor.c rgb_ycc_convert) */

static void bgr_to_ycc(const uint8_t *p, int *y, int *cb, int *cr) {
    int b = p[0], g = p[1], r = p[2];
    *y = (19595 * r + 38470 * g + 7471 * b + 32768) >> 16;
    *cb = (-11059 * r - 21709 * g + 32768 * b + (128 << 16) + 32767) >> 16;
    *cr = (32768 * r - 27439 * g - 5329 * b + (128 << 16) + 32767) >> 16;
}

/* ------------------------------------------------------------------ A.4 FDCT (jfdctint.c jpeg_fdct_islow) */

#define DESCALE(x, n) (((x) + (1 << ((n)-1))) >> (n))
#define F_0_298 2446
#define F_0_390 3196
#define F_0_541 4433
#define F_0_765 6270
#define F_0_899 7373
#define F_1_175 9633
#define F_1_501 12299
#define F_1_847 15137
#define F_1_961 16069
#define F_2_053 16819
#define F_2_562 20995
#define F_3_072 25172

static void fdct_1d(const int *d, int stride, int *o, int pass2) {
    int d0 = d[0], d1 = d[stride], d2 = d[2 * stride], d3 = d[3 * stride], d4 = d[4 * stride], d5 = d[5 * stride],
        d6 = d[6 * stride], d7 = d[7 * stride];
    int t0 = d0 + d7, t7 = d0 - d7, t1 = d1 + d6, t6 = d1 - d6, t2 = d2 + d5, t5 = d2 - d5, t3 = d3 + d4, t4 = d3 - d4;
    int t10 = t0 + t3, t13 = t0 - t3, t11 = t1 + t2, t12 = t1 - t2;
    int sh = pass2 ? 15 : 11;
    int o0, o4;
    if (!pass2) { o0 = (t10 + t11) << 2; o4 = (t10 - t11) << 2; }
    else { o0 = DESCALE(t10 + t11, 2); o4 = DESCALE(t10 - t11, 2); }
    int z1 = (t12 + t13) * F_0_541;
    int o2 = DESCALE(z1 + t13 * F_0_765, sh);
    int o6 = DESCALE(z1 - t12 * F_1_847, sh);
    z1 = t4 + t7; int z2 = t5 + t6, z3 = t4 + t6, z4 = t5 + t7;
    int z5 = (z3 + z4) * F_1_175;
    t4 *= F_0_298; t5 *= F_2_053; t6 *= F_3_072; t7 *= F_1_501;
    z1 *= -F_0_899; z2 *= -F_2_562; z3 = z3 * (-F_1_961) + z5; z4 = z4 * (-F_0_390) + z5;
    int o7 = DESCALE(t4 + z1 + z3, sh), o5 = DESCALE(t5 + z2 + z4, sh), o3 = DESCALE(t6 + z2 + z3, sh),
        o1 = DESCALE(t7 + z1 + z4, sh);
    o[0] = o0; o[stride] = o1; o[2 * stride] = o2; o[3 * stride] = o3; o[4 * stride] = o4; o[5 * stride] = o5;
    o[6 * stride] = o6; o[7 * stride] = o7;
}

static void fdct_block(const uint8_t *s, int stride, int *out /* natural order, 64 */) {
    int w[64];
    for (int r = 0; r < 8; r++)
        for (int c = 0; c < 8; c++) w[r * 8 + c] = (int)s[r * stride + c] - 128;
    for (int r = 0; r < 8; r++) fdct_1d(w + r * 8, 1, w + r * 8, 0);
    for (int c = 0; c < 8; c++) fdct_1d(w + c, 8, w + c, 1);
    memcpy(out, w, sizeof(w));
}

/* A.5 quantisation (jcdctmgr.c quantize): divisor 8*q, round half away from zero */
static int16_t quantise(int c, int q) {
    int d = 8 * q;
    int a = c < 0 ? -c : c;
    a = (a + (d >> 1)) / d;
    return (int16_t)(c < 0 ? -a : a);
}

/* ------------------------------------------------------------------ A.3 padding + downsampling, A.6 block order / dummy blocks */

int orc_forward(const uint8_t *bgr, size_t step, int W, int H, int css, int quality, int16_t *coef) {
    orc_geom g;
    if (orc_geometry(W, H, css, &g)) return -1;
    uint16_t qt[2][64];
    orc_quant_tables(quality, qt);

    /* full-resolution YCbCr planes */
    size_t npx = (size_t)W * H;
    uint8_t *full[3];
    for (int c = 0; c < 3; c++) { full[c] = (uint8_t *)malloc(npx); if (!full[c]) return -2; }
    for (int y = 0; y < H; y++)
        for (int x = 0; x < W; x++) {
            int yy, cb, cr;
            bgr_to_ycc(bgr + (size_t)y * step + (size_t)x * 3, &yy, &cb, &cr);
            full[0][(size_t)y * W + x] = (uint8_t)yy; full[1][(size_t)y * W + x] = (uint8_t)cb;
            full[2][(size_t)y * W + x] = (uint8_t)cr;
        }

    /* per-component padded, downsampled planes: width wib*8, height mcuy*v*8 */
    uint8_t *pl[3]; int pw[3], ph[3];
    for (int c = 0; c < 3; c++) {
        int h = c ? 1 : g.hs, v = c ? 1 : g.vs;
        int hx = g.hs / h, vx = g.vs / v;
        pw[c] = g.wib[c] * 8; ph[c] = g.mcuy * v * 8;
        pl[c] = (uint8_t *)malloc((size_t)pw[c] * ph[c]);
        if (!pl[c]) return -2;
        int dh = g.dh[c]; /* = ceil(H/vx): rows that come out of the downsampler after step (1) */
        for (int r = 0; r < ph[c]; r++) {
            int rs = r < dh ? r : dh - 1; /* step (4): replicate last downsampled row */
            for (int j = 0; j < pw[c]; j++) {
                int sum = 0;
                for (int dy = 0; dy < vx; dy++) {
                    int yy = rs * vx + dy; if (yy > H - 1) yy = H - 1;     /* step (1) */
                    for (int dx = 0; dx < hx; dx++) {
                        int xx = j * hx + dx; if (xx > W - 1) xx = W - 1;  /* step (2) */
                        sum += full[c][(size_t)yy * W + xx];
                    }
                }
                int o;
                if (hx == 1 && vx == 1) o = sum;
                else if (hx == 2 && vx == 1) o = (sum + (j & 1)) >> 1;        /* h2v1_downsample: bias 0,1,0,1 */
                else if (hx == 2 && vx == 2) o = (sum + 1 + (j & 1)) >> 2;    /* h2v2_downsample: bias 1,2,1,2 */
                else { int n = hx * vx; o = (sum + n / 2) / n; }              /* int_downsample */
                pl[c][(size_t)r * pw[c] + j] = (uint8_t)o;
            }
        }
    }

    /* blocks in scan order */
    int nat[64];
    for (int my = 0; my < g.mcuy; my++)
        for (int mx = 0; mx < g.mcux; mx++) {
            int16_t *mcu = coef + ((size_t)my * g.mcux + mx) * g.bpm * 64;
            int blkn = 0;
            for (int c = 0; c < 3; c++) {
                int h = c ? 1 : g.hs, v = c ? 1 : g.vs;
                const uint16_t *q = qt[c ? 1 : 0];
                for (int by = 0; by < v; by++) {
                    int brow = my * v + by;
                    for (int bx = 0; bx < h; bx++, blkn++) {
                        int bcol = mx * h + bx;
                        int16_t *blk = mcu + blkn * 64;
                        if (brow < g.hib[c] && bcol < g.wib[c]) {
                            fdct_block(pl[c] + (size_t)brow * 8 * pw[c] + (size_t)bcol * 8, pw[c], nat);
                            for (int k = 0; k < 64; k++) blk[k] = quantise(nat[ZIGZAG[k]], q[ZIGZAG[k]]);
                        } else if (brow < g.hib[c]) { /* right-edge dummy: DC of the block to the left */
                            memset(blk, 0, 128); blk[0] = (blk - 64)[0];
                        } else {                      /* bottom dummy row: DC of last block of the row above */
                            memset(blk, 0, 128); blk[0] = (mcu + (blkn - bx - 1) * 64)[0];
                        }
                    }
                }
            }
        }
    for (int c = 0; c < 3; c++) { free(full[c]); free(pl[c]); }
    return 0;
}

/* ------------------------------------------------------------------ scan-order helpers */

/* bpm 1 (one component): every block is the last component's, so its tables are slots 2 / 3 (DC1 / AC1) */
static int comp_of_block(int blkn, int bpm) { return blkn < bpm - 2 ? 0 : (blkn == bpm - 2 ? 1 : 2); }
static int nbits_of(int v) { int a = v < 0 ? -v : v, n = 0; while (a) { n++; a >>= 1; } return n; }

/* jchuff.c htest_one_block */
void orc_histogram(const int16_t *coef, long long nblocks, int bpm, const int16_t *pred_in, uint32_t hist[4][257]) {
    int pred[3] = {0, 0, 0};
    if (pred_in) { pred[0] = pred_in[0]; pred[1] = pred_in[1]; pred[2] = pred_in[2]; }
    memset(hist, 0, sizeof(uint32_t) * 4 * 257);
    for (long long b = 0; b < nblocks; b++) {
        const int16_t *blk = coef + b * 64;
        int c = comp_of_block((int)(b % bpm), bpm);
        int t = c ? 1 : 0;
        int diff = blk[0] - pred[c]; pred[c] = blk[0];
        hist[2 * t][nbits_of(diff)]++;
        int r = 0;
        for (int k = 1; k < 64; k++) {
            if (blk[k] == 0) { r++; continue; }
            while (r > 15) { hist[2 * t + 1][0xF0]++; r -= 16; }
            hist[2 * t + 1][(r << 4) + nbits_of(blk[k])]++;
            r = 0;
        }
        if (r > 0) hist[2 * t + 1][0]++;
    }
}

/* ------------------------------------------------------------------ A.7 jchuff.c jpeg_gen_optimal_table */

int orc_gen_optimal_table(const uint32_t freq_in[257], uint8_t bits_out[17], uint8_t huffval[256]) {
    long freq[257]; int codesize[257], others[257]; int bits[33];
    for (int i = 0; i < 257; i++) { freq[i] = (long)freq_in[i]; codesize[i] = 0; others[i] = -1; }
    memset(bits, 0, sizeof(bits));
    freq[256] = 1;
    for (;;) {
        int c1 = -1, c2 = -1; long v = 1000000000L;
        for (int i = 0; i <= 256; i++) if (freq[i] && freq[i] <= v) { v = freq[i]; c1 = i; }
        v = 1000000000L;
        for (int i = 0; i <= 256; i++) if (freq[i] && freq[i] <= v && i != c1) { v = freq[i]; c2 = i; }
        if (c2 < 0) break;
        freq[c1] += freq[c2]; freq[c2] = 0;
        codesize[c1]++; while (others[c1] >= 0) { c1 = others[c1]; codesize[c1]++; }
        others[c1] = c2;
        codesize[c2]++; while (others[c2] >= 0) { c2 = others[c2]; codesize[c2]++; }
    }
    for (int i = 0; i <= 256; i++) if (codesize[i]) { if (codesize[i] > 32) return -1; bits[codesize[i]]++; }
    for (int i = 32; i > 16; i--)
        while (bits[i] > 0) {
            int j = i - 2; while (bits[j] == 0) j--;
            bits[i] -= 2; bits[i - 1]++; bits[j + 1] += 2; bits[j]--;
        }
    int i = 16; while (bits[i] == 0) i--;
    bits[i]--;
    bits_out[0] = 0;
    for (int k = 1; k <= 16; k++) bits_out[k] = (uint8_t)bits[k];
    int p = 0;
    memset(huffval, 0, 256);
    for (int len = 1; len <= 32; len++)
        for (int j = 0; j <= 255; j++) if (codesize[j] == len) huffval[p++] = (uint8_t)j;
    return p;
}

int orc_std_table(int idx, uint8_t bits[17], uint8_t huffval[256]) {
    memset(huffval, 0, 256);
    switch (idx) {
    case 0: memcpy(bits, STD_DC_LUMA_BITS, 17); memcpy(huffval, STD_DC_VAL, 12); return 12;
    case 1: memcpy(bits, STD_AC_LUMA_BITS, 17); memcpy(huffval, STD_AC_LUMA_VAL, 162); return 162;
    case 2: memcpy(bits, STD_DC_CHROMA_BITS, 17); memcpy(huffval, STD_DC_VAL, 12); return 12;
    case 3: memcpy(bits, STD_AC_CHROMA_BITS, 17); memcpy(huffval, STD_AC_CHROMA_VAL, 162); return 162;
    }
    return -1;
}

/* Annex C / jchuff.c jpeg_make_c_derived_tbl */
void orc_derive_codes(const uint8_t bits[17], const uint8_t huffval[256], uint16_t code[256], uint8_t size[256]) {
    memset(code, 0, 512); memset(size, 0, 256);
    int p = 0; unsigned c = 0;
    for (int l = 1; l <= 16; l++) {
        for (int i = 0; i < bits[l]; i++) { code[huffval[p]] = (uint16_t)c; size[huffval[p]] = (uint8_t)l; p++; c++; }
        c <<= 1;
    }
}

/* ------------------------------------------------------------------ A.6 entropy coding (jchuff.c encode_one_block) */

typedef struct { uint8_t *out; size_t cap; uint64_t nbits; int overflow; } bitw;
static void put_bits(bitw *w, unsigned code, int size) {
    for (int i = size - 1; i >= 0; i--) {
        uint64_t pos = w->nbits++;
        if ((pos >> 3) >= w->cap) { w->overflow = 1; continue; }
        if ((code >> i) & 1) w->out[pos >> 3] |= (uint8_t)(0x80 >> (pos & 7));
    }
}

int orc_entropy_bits(const int16_t *coef, long long nblocks, int bpm, const int16_t *pred_in,
                     const uint8_t bits[4][17], const uint8_t vals[4][256], uint8_t *out, size_t cap, uint64_t *nbits) {
    uint16_t code[4][256]; uint8_t size[4][256];
    for (int t = 0; t < 4; t++) orc_derive_codes(bits[t], vals[t], code[t], size[t]);
    int pred[3] = {0, 0, 0};
    if (pred_in) { pred[0] = pred_in[0]; pred[1] = pred_in[1]; pred[2] = pred_in[2]; }
    memset(out, 0, cap);
    bitw w = {out, cap, 0, 0};
    for (long long b = 0; b < nblocks; b++) {
        const int16_t *blk = coef + b * 64;
        int c = comp_of_block((int)(b % bpm), bpm);
        int dt = c ? 2 : 0, at = dt + 1;
        int diff = blk[0] - pred[c]; pred[c] = blk[0];
        int n = nbits_of(diff);
        int v = diff < 0 ? diff - 1 : diff;
        put_bits(&w, code[dt][n], size[dt][n]);
        if (n) put_bits(&w, (unsigned)v & ((1u << n) - 1), n);
        int r = 0;
        for (int k = 1; k < 64; k++) {
            int x = blk[k];
            if (x == 0) { r++; continue; }
            while (r > 15) { put_bits(&w, code[at][0xF0], size[at][0xF0]); r -= 16; }
            n = nbits_of(x);
            v = x < 0 ? x - 1 : x;
            put_bits(&w, code[at][(r << 4) + n], size[at][(r << 4) + n]);
            put_bits(&w, (unsigned)v & ((1u << n) - 1), n);
            r = 0;
        }
        if (r > 0) put_bits(&w, code[at][0], size[at][0]);
    }
    *nbits = w.nbits;
    return w.overflow ? -1 : 0;
}

size_t orc_stuff(const uint8_t *in, uint64_t nbits, uint8_t *out, size_t cap) {
    size_t nbytes = (size_t)((nbits + 7) >> 3), o = 0;
    for (size_t i = 0; i < nbytes; i++) {
        uint8_t b = in[i];
        if (i == nbytes - 1 && (nbits & 7)) b |= (uint8_t)(0xFF >> (nbits & 7)); /* pad with 1-bits */
        if (o < cap) out[o] = b;
        o++;
        if (b == 0xFF) { if (o < cap) out[o] = 0; o++; }
    }
    return o;
}

/* ------------------------------------------------------------------ A.8 markers (jcmarker.c) */

typedef struct { uint8_t *out; size_t n, cap; } bytew;   /* counts past cap without writing */
static void put(bytew *w, int b) { if (w->n < w->cap) w->out[w->n] = (uint8_t)b; w->n++; }
static void put16(bytew *w, int v) { put(w, v >> 8); put(w, v & 255); }

/* SOI, JFIF APP0, one DQT per table in use, SOF (marker byte `sof`) with component ids 1, 2, 3 */
static void put_frame(bytew *w, int sof, const orc_geom *g, const uint16_t qt[2][64]) {
    static const uint8_t app0[18] = {0xFF, 0xE0, 0, 16, 'J', 'F', 'I', 'F', 0, 1, 1, 0, 0, 1, 0, 1, 0, 0};
    const int nc = g->css == ORC_CSS_GRAY ? 1 : 3;
    put16(w, 0xFFD8);
    for (int i = 0; i < 18; i++) put(w, app0[i]);
    for (int t = 0; t < (nc == 1 ? 1 : 2); t++) {
        put16(w, 0xFFDB); put16(w, 67); put(w, t);
        for (int k = 0; k < 64; k++) put(w, qt[t][ZIGZAG[k]]);
    }
    put16(w, 0xFF00 | sof); put16(w, 8 + 3 * nc); put(w, 8); put16(w, g->H); put16(w, g->W); put(w, nc);
    for (int c = 0; c < nc; c++) { put(w, c + 1); put(w, c ? 0x11 : (g->hs << 4) | g->vs); put(w, c ? 1 : 0); }
}
static void put_dht(bytew *w, int tc_th, const uint8_t bits[17], const uint8_t *vals) {
    int ns = 0; for (int l = 1; l <= 16; l++) ns += bits[l];
    put16(w, 0xFFC4); put16(w, 19 + ns); put(w, tc_th);
    for (int l = 1; l <= 16; l++) put(w, bits[l]);
    for (int i = 0; i < ns; i++) put(w, vals[i]);
}
/* SOS of components comp[0..n-1] (ids comp + 1), table selector bytes sel[] */
static void put_sos(bytew *w, int n, const int comp[], const int sel[], int Ss, int Se, int Ah_Al) {
    put16(w, 0xFFDA); put16(w, 6 + 2 * n); put(w, n);
    for (int i = 0; i < n; i++) { put(w, comp[i] + 1); put(w, sel[i]); }
    put(w, Ss); put(w, Se); put(w, Ah_Al);
}
/* a one-scan baseline file: the frame, DHT DC0 AC0 (DC1 AC1) from bits / vals [0..3] ([0..1] for one component), DRI
 * when there are restart intervals (write_scan_header: after the scan's DHTs, before SOS), SOS */
static void put_baseline_headers(bytew *w, const orc_geom *g, const uint16_t qt[2][64], const uint8_t bits[][17],
                                 const uint8_t vals[][256], int ri) {
    static const int comp[3] = {0, 1, 2}, sel[3] = {0x00, 0x11, 0x11};
    const int nc = g->css == ORC_CSS_GRAY ? 1 : 3;
    put_frame(w, 0xC0, g, qt);
    for (int t = 0; t < 2 * (nc == 1 ? 1 : 2); t++) put_dht(w, (t & 1) << 4 | t >> 1, bits[t], vals[t]);
    if (ri) { put16(w, 0xFFDD); put16(w, 4); put16(w, ri); }
    put_sos(w, nc, comp, sel, 0, 63, 0);
}

size_t orc_headers(int W, int H, int css, const uint16_t qt[2][64], const uint8_t bits[4][17],
                   const uint8_t vals[4][256], uint8_t *out, size_t cap) {
    orc_geom g; if (orc_geometry(W, H, css, &g)) return 0;
    bytew w = {out, 0, cap};
    put_baseline_headers(&w, &g, qt, bits, vals, 0);
    return w.n > cap ? 0 : w.n;
}

/* one component (jccolor.c grayscale_convert): the samples as they stand, edges replicated to whole blocks
 * (jcsample.c expand_right_edge, jcprepct.c), quantised with the luma table */
static void forward_gray(const uint8_t *gray, size_t step, const orc_geom *g, const uint16_t qt[64], int16_t *coef) {
    int nat[64]; uint8_t blk8[64];
    for (int by = 0; by < g->mcuy; by++)
        for (int bx = 0; bx < g->mcux; bx++) {
            for (int r = 0; r < 8; r++)
                for (int c = 0; c < 8; c++) {
                    int y = by * 8 + r, x = bx * 8 + c;
                    blk8[r * 8 + c] = gray[(size_t)(y < g->H ? y : g->H - 1) * step + (x < g->W ? x : g->W - 1)];
                }
            fdct_block(blk8, 8, nat);
            int16_t *blk = coef + ((size_t)by * g->mcux + bx) * 64;
            for (int k = 0; k < 64; k++) blk[k] = quantise(nat[ZIGZAG[k]], qt[ZIGZAG[k]]);
        }
}

/* The baseline encoder, three components (BGR pixels) or one (gray samples, g->css == ORC_CSS_GRAY: the stream's DC0 /
 * AC0 tables are slots 2 / 3 of orc_histogram and orc_entropy_bits). Restart intervals (jchuff.c
 * emit_restart, jcmarker.c emit_dri): every `ri` MCUs (0 = none; a one-component MCU is one block) the bit buffer is
 * flushed (1-padding to a byte boundary, stuffing applies to the padded byte), RSTn (n = 0..7 cycling) is written
 * unstuffed and the DC predictors return to 0; no marker follows the last interval. Symbol statistics use the same
 * predictor resets. */
static int encode_baseline(const uint8_t *px, size_t step, const orc_geom *g, int quality, int optimize, int ri,
                           uint8_t *out, size_t cap, size_t *len) {
    if (g->W > 65535 || g->H > 65535 || ri < 0 || ri > 65535) return -1;
    const int t0 = g->bpm == 1 ? 2 : 0;   /* the slots of the stream's tables: t0 .. 3 */
    const long long nmcu = (long long)g->mcux * g->mcuy, iv = ri ? ri : nmcu;
    int16_t *coef = (int16_t *)malloc((size_t)g->nblocks * 128);
    uint8_t *raw = (uint8_t *)malloc((size_t)iv * g->bpm * 208 + 16);   /* worst case 64 coefs * 26 bits */
    uint16_t qt[2][64]; orc_quant_tables(quality, qt);
    uint8_t bits[4][17], vals[4][256];
    memset(bits, 0, sizeof(bits)); memset(vals, 0, sizeof(vals));
    int rc = coef && raw ? 0 : -2;
    if (!rc) {
        if (g->bpm == 1) forward_gray(px, step, g, qt[0], coef);
        else rc = orc_forward(px, step, g->W, g->H, g->css, quality, coef);
    }
    if (!rc && optimize) {
        uint32_t hist[4][257], h1[4][257];
        memset(hist, 0, sizeof(hist));
        for (long long m0 = 0; m0 < nmcu; m0 += iv) {
            orc_histogram(coef + m0 * g->bpm * 64, (nmcu - m0 < iv ? nmcu - m0 : iv) * g->bpm, g->bpm, NULL, h1);
            for (int t = 0; t < 4; t++) for (int i = 0; i < 257; i++) hist[t][i] += h1[t][i];
        }
        for (int t = t0; t < 4; t++) if (orc_gen_optimal_table(hist[t], bits[t], vals[t]) < 0) rc = -3;
    } else if (!rc) {
        for (int t = t0; t < 4; t++) orc_std_table(t - t0, bits[t], vals[t]);
    }
    bytew w = {out, 0, cap};
    if (!rc) {
        put_baseline_headers(&w, g, qt, (const uint8_t(*)[17])bits + t0, (const uint8_t(*)[256])vals + t0, ri);
        if (w.n > cap) rc = -4;
    }
    size_t o = w.n;
    int rstn = 0;
    for (long long m0 = 0; !rc && m0 < nmcu; m0 += iv) {
        uint64_t nbits = 0;
        if (orc_entropy_bits(coef + m0 * g->bpm * 64, (nmcu - m0 < iv ? nmcu - m0 : iv) * g->bpm, g->bpm, NULL,
                             (const uint8_t(*)[17])bits, (const uint8_t(*)[256])vals, raw, (size_t)iv * g->bpm * 208 + 16,
                             &nbits)) { rc = -5; break; }
        o += orc_stuff(raw, nbits, out + o, cap > o ? cap - o : 0);
        if (o + 2 > cap) { rc = -6; break; }
        if (m0 + iv < nmcu) { out[o++] = 0xFF; out[o++] = (uint8_t)(0xD0 + rstn); rstn = (rstn + 1) & 7; }
    }
    free(coef); free(raw);
    if (rc) return rc;
    out[o++] = 0xFF; out[o++] = 0xD9;
    *len = o;
    return 0;
}

int orc_encode(const uint8_t *bgr, size_t step, int W, int H, int css, int quality, int optimize, uint8_t *out,
               size_t cap, size_t *len) {
    return orc_encode_rst(bgr, step, W, H, css, quality, optimize, 0, out, cap, len);
}

int orc_encode_rst(const uint8_t *px, size_t step, int W, int H, int css, int quality, int optimize, int ri,
                   uint8_t *out, size_t cap, size_t *len) {
    orc_geom g;
    if (css == ORC_CSS_GRAY && W > 0 && H > 0) layout(W, H, css, &g);
    else if (orc_geometry(W, H, css, &g)) return -1;
    return encode_baseline(px, step, &g, quality, optimize, ri < 0 ? 0 : ri, out, cap, len);
}

/* scan parameters and the scan-order index of block (bx, by) of component c (shared by both progressive halves) */
typedef struct { int ncomp, comp[3], td[3], ta[3], Ss, Se, Ah, Al; } pscan;

static size_t block_index(const orc_geom *g, int c, int bx, int by) {
    int h = c ? 1 : g->hs, v = c ? 1 : g->vs;
    int mx = bx / h, my = by / v;
    int blkn = c ? g->bpm - 3 + c : (by % v) * h + (bx % h);
    return ((size_t)my * g->mcux + mx) * g->bpm + blkn;
}

/* ------------------------------------------------------------------ progressive (SOF2) encode: jcphuff.c
 * jpeg_simple_progression's 10-scan script for YCbCr (jcparam.c), every scan with its own optimal Huffman tables
 * (progressive mode forces optimize_coding): each scan is walked twice, first counting symbols, then emitting. */
typedef struct {
    int gather;                 /* pass 1: count symbols; pass 2: emit */
    uint32_t count[257];        /* the scan's AC table, or (DC scans) indexed through cnt_dc */
    uint32_t cnt_dc[2][257];
    uint16_t code[2][256]; uint8_t size[2][256];   /* [0] = DC/AC luma table of this scan, [1] = chroma */
    bitw w;
    unsigned eobrun; int be; uint8_t bebuf[1024];
} penc;

static void p_sym(penc *e, int tbl, int sym, int is_dc) {
    if (e->gather) { if (is_dc) e->cnt_dc[tbl][sym]++; else e->count[sym]++; }
    else put_bits(&e->w, e->code[tbl][sym], e->size[tbl][sym]);
}
static void p_bits(penc *e, unsigned v, int n) { if (!e->gather && n) put_bits(&e->w, v & ((1u << n) - 1), n); }
static void p_buffered(penc *e, const uint8_t *b, int n) { if (!e->gather) for (int i = 0; i < n; i++) put_bits(&e->w, b[i], 1); }
static void p_eobrun(penc *e, int tbl) {
    if (e->eobrun > 0) {
        unsigned t = e->eobrun; int nb = 0;
        while (t >>= 1) nb++;
        p_sym(e, tbl, nb << 4, 0);
        if (nb) p_bits(e, e->eobrun, nb);
        e->eobrun = 0;
        p_buffered(e, e->bebuf, e->be);
        e->be = 0;
    }
}

static void p_ac_first(penc *e, int tbl, const int16_t *blk, int Ss, int Se, int Al) {
    int r = 0;
    for (int k = Ss; k <= Se; k++) {
        int t = blk[k], t2;
        if (t == 0) { r++; continue; }
        if (t < 0) { t = -t; t >>= Al; t2 = ~t; } else { t >>= Al; t2 = t; }
        if (t == 0) { r++; continue; }
        if (e->eobrun > 0) p_eobrun(e, tbl);
        while (r > 15) { p_sym(e, tbl, 0xF0, 0); r -= 16; }
        int nb = nbits_of(t);
        p_sym(e, tbl, (r << 4) + nb, 0);
        p_bits(e, (unsigned)t2, nb);
        r = 0;
    }
    if (r > 0) { e->eobrun++; if (e->eobrun == 0x7FFF) p_eobrun(e, tbl); }
}

static void p_ac_refine(penc *e, int tbl, const int16_t *blk, int Ss, int Se, int Al) {
    int absv[64], EOB = 0;
    for (int k = Ss; k <= Se; k++) {
        int t = blk[k]; if (t < 0) t = -t;
        t >>= Al; absv[k] = t;
        if (t == 1) EOB = k;
    }
    int r = 0, br = 0;
    uint8_t *brbuf = e->bebuf + e->be;
    for (int k = Ss; k <= Se; k++) {
        int t = absv[k];
        if (t == 0) { r++; continue; }
        while (r > 15 && k <= EOB) {
            p_eobrun(e, tbl);
            p_sym(e, tbl, 0xF0, 0);
            r -= 16;
            p_buffered(e, brbuf, br);
            brbuf = e->bebuf; br = 0;
        }
        if (t > 1) { brbuf[br++] = (uint8_t)(t & 1); continue; }
        p_eobrun(e, tbl);
        p_sym(e, tbl, (r << 4) + 1, 0);
        p_bits(e, blk[k] < 0 ? 0u : 1u, 1);
        p_buffered(e, brbuf, br);
        brbuf = e->bebuf; br = 0;
        r = 0;
    }
    if (r > 0 || br > 0) {
        e->eobrun++;
        e->be += br;
        if (e->eobrun == 0x7FFF || e->be > 1000 - 64 + 1) p_eobrun(e, tbl);
    }
}

/* one scan, one pass (gather or emit) over the coefficient array */
static void p_scan(penc *e, const orc_geom *g, const int16_t *coef, const pscan *sc, int ri) {
    int pred[3] = {0, 0, 0};
    (void)ri;   /* restart intervals: not restated for progressive encode */
    e->eobrun = 0; e->be = 0;
    if (sc->ncomp > 1) {
        for (long long mi = 0; mi < (long long)g->mcux * g->mcuy; mi++) {
            for (int i = 0; i < sc->ncomp; i++) {
                int c = sc->comp[i], nb = c ? 1 : g->hs * g->vs, b0 = c ? g->bpm - 3 + c : 0, tblc = c ? 1 : 0;
                for (int b = 0; b < nb; b++) {
                    const int16_t *blk = coef + ((size_t)mi * g->bpm + b0 + b) * 64;
                    if (sc->Ah == 0) {
                        int t2 = blk[0] >> sc->Al, d = t2 - pred[c];
                        pred[c] = t2;
                        int n = nbits_of(d), v = d < 0 ? d - 1 : d;
                        p_sym(e, tblc, n, 1);
                        p_bits(e, (unsigned)v, n);
                    } else {
                        p_bits(e, (unsigned)(blk[0] >> sc->Al) & 1u, 1);
                    }
                }
            }
        }
    } else {
        int c = sc->comp[0], tblc = c ? 1 : 0;
        for (int by = 0; by < g->hib[c]; by++)
            for (int bx = 0; bx < g->wib[c]; bx++) {
                const int16_t *blk = coef + block_index(g, c, bx, by) * 64;
                if (sc->Ss == 0) {
                    if (sc->Ah == 0) {
                        int t2 = blk[0] >> sc->Al, d = t2 - pred[c];
                        pred[c] = t2;
                        int n = nbits_of(d), v = d < 0 ? d - 1 : d;
                        p_sym(e, tblc, n, 1);
                        p_bits(e, (unsigned)v, n);
                    } else p_bits(e, (unsigned)(blk[0] >> sc->Al) & 1u, 1);
                } else if (sc->Ah == 0) p_ac_first(e, tblc, blk, sc->Ss, sc->Se, sc->Al);
                else p_ac_refine(e, tblc, blk, sc->Ss, sc->Se, sc->Al);
            }
        p_eobrun(e, tblc);
    }
}

int orc_encode_progressive(const uint8_t *bgr, size_t step, int W, int H, int css, int quality, uint8_t *out,
                           size_t cap, size_t *len) {
    orc_geom g; if (orc_geometry(W, H, css, &g)) return -1;
    if (W > 65535 || H > 65535) return -1;
    int16_t *coef = (int16_t *)malloc((size_t)g.nblocks * 128);
    if (!coef) return -2;
    int rc = orc_forward(bgr, step, W, H, css, quality, coef);
    if (rc) { free(coef); return rc; }
    uint16_t qt[2][64]; orc_quant_tables(quality, qt);
    bytew w = {out, 0, cap};
    put_frame(&w, 0xC2, &g, qt);
    /* jcparam.c jpeg_simple_progression, YCbCr: {comps, Ss, Se, Ah, Al} */
    static const int script[10][5] = {{-1, 0, 0, 0, 1}, {0, 1, 5, 0, 2}, {2, 1, 63, 0, 1}, {1, 1, 63, 0, 1}, {0, 6, 63, 0, 2},
                                      {0, 1, 63, 2, 1}, {-1, 0, 0, 1, 0}, {2, 1, 63, 1, 0}, {1, 1, 63, 1, 0}, {0, 1, 63, 1, 0}};
    size_t raw_cap = (size_t)g.nblocks * 208 + 64;
    uint8_t *raw = (uint8_t *)malloc(raw_cap);
    penc *e = (penc *)malloc(sizeof(penc));
    if (!raw || !e) { free(coef); free(raw); free(e); return -2; }
    for (int si = 0; si < 10; si++) {
        pscan sc; memset(&sc, 0, sizeof(sc));
        if (script[si][0] < 0) { sc.ncomp = 3; sc.comp[0] = 0; sc.comp[1] = 1; sc.comp[2] = 2; }
        else { sc.ncomp = 1; sc.comp[0] = script[si][0]; }
        sc.Ss = script[si][1]; sc.Se = script[si][2]; sc.Ah = script[si][3]; sc.Al = script[si][4];
        const int is_dc = sc.Ss == 0, need_tbl = !(is_dc && sc.Ah != 0);
        memset(e, 0, sizeof(*e));
        uint8_t bits[2][17], vals[2][256];
        if (need_tbl) {
            e->gather = 1;
            p_scan(e, &g, coef, &sc, 0);
            for (int t = 0; t < 2; t++) {
                const uint32_t *cnt = is_dc ? e->cnt_dc[t] : e->count;
                int used = is_dc ? 1 : (t == (sc.comp[0] ? 1 : 0));
                if (!used) continue;
                if (orc_gen_optimal_table(cnt, bits[t], vals[t]) < 0) { free(coef); free(raw); free(e); return -3; }
                orc_derive_codes(bits[t], vals[t], e->code[t], e->size[t]);
                put_dht(&w, (is_dc ? 0x00 : 0x10) | t, bits[t], vals[t]);
            }
        }
        int sel[3];
        for (int i = 0; i < sc.ncomp; i++) { int t = sc.comp[i] ? 1 : 0; sel[i] = is_dc ? (sc.Ah == 0 ? t << 4 : 0) : t; }
        put_sos(&w, sc.ncomp, sc.comp, sel, sc.Ss, sc.Se, (sc.Ah << 4) | sc.Al);
        e->gather = 0;
        memset(raw, 0, raw_cap);
        e->w.out = raw; e->w.cap = raw_cap; e->w.nbits = 0; e->w.overflow = 0;
        p_scan(e, &g, coef, &sc, 0);
        if (e->w.overflow) { free(coef); free(raw); free(e); return -5; }
        w.n += orc_stuff(raw, e->w.nbits, w.n < cap ? out + w.n : out, w.n < cap ? cap - w.n : 0);
    }
    put16(&w, 0xFFD9);
    free(coef); free(raw); free(e);
    if (w.n > cap) return -6;
    *len = w.n;
    return 0;
}

/* ------------------------------------------------------------------ decoder: Huffman (jdhuff.c) */

static int rd16(const uint8_t *p) { return (p[0] << 8) | p[1]; }

typedef struct { int mincode[17], maxcode[18], valptr[17]; const uint8_t *vals; } dtbl;
static void make_dtbl(const uint8_t bits[17], const uint8_t *vals, dtbl *t) {
    int code = 0, p = 0;
    for (int l = 1; l <= 16; l++) {
        t->valptr[l] = p; t->mincode[l] = code;
        p += bits[l]; code += bits[l];
        t->maxcode[l] = bits[l] ? code - 1 : -1;
        code <<= 1;
    }
    t->maxcode[17] = 0x7fffffff; t->vals = vals;
}
/* insufficient: a bit past the data (a marker or the end of the segment) was read; jdhuff.c jpeg_fill_bit_buffer then
 * feeds zero bits and sets the entropy decoder's insufficient_data */
typedef struct { const uint8_t *d; size_t n, pos; uint32_t acc; int cnt; int marker; int insufficient; } bitr;
static int get_bit(bitr *r) {
    if (r->cnt == 0) {
        uint8_t b = 0;
        if (r->pos < r->n && !r->marker) {
            b = r->d[r->pos];
            if (b == 0xFF) {   /* jdhuff.c fill_bit_buffer: any number of 0xFF, then 00 (data) or a marker */
                size_t q = r->pos + 1;
                while (q < r->n && r->d[q] == 0xFF) q++;
                uint8_t b2 = q < r->n ? r->d[q] : 0xD9;
                if (b2 == 0) r->pos = q + 1; else { r->marker = b2; r->pos = q - 1; b = 0; r->insufficient = 1; }
            } else r->pos++;
        } else r->insufficient = 1;
        r->acc = b; r->cnt = 8;
    }
    r->cnt--;
    return (r->acc >> r->cnt) & 1;
}
static int get_bits(bitr *r, int n) { int v = 0; while (n--) v = (v << 1) | get_bit(r); return v; }
static int decode_sym(bitr *r, const dtbl *t) {
    int code = 0;
    for (int l = 1; l <= 16; l++) {
        code = (code << 1) | get_bit(r);
        if (t->maxcode[l] >= 0 && code <= t->maxcode[l] && code >= t->mincode[l]) return t->vals[t->valptr[l] + code - t->mincode[l]];
    }
    return 0;
}
static int extend(int v, int n) { return n == 0 ? 0 : (v < (1 << (n - 1)) ? v - (1 << n) + 1 : v); }

/* the end of a scan's entropy-coded data: the first marker that is not RSTn / stuffed zero, less the fill bytes (0xFF)
 * in front of it */
static size_t entropy_end(const uint8_t *jpg, size_t len, size_t e0) {
    size_t e = e0;
    while (e + 1 < len) {
        if (jpg[e] == 0xFF && jpg[e + 1] != 0x00 && jpg[e + 1] != 0xFF && !(jpg[e + 1] >= 0xD0 && jpg[e + 1] <= 0xD7)) break;
        e++;
    }
    if (e + 1 >= len) e = len;
    while (e > e0 && jpg[e - 1] == 0xFF) e--;
    return e;
}

/* jdhuff.c / jdphuff.c process_restart. Where the data ends instead of an RSTn (a cut file), insufficient_data stays as
 * it is: the rest of a progressive scan is left alone, except that an interval that ended cleanly lets the next one
 * decode one MCU of zero bits before it runs out */
static void prog_restart(bitr *r, int pred[3], int *eobrun) {
    r->cnt = 0;
    while (!r->marker && r->pos + 1 < r->n && r->d[r->pos] == 0xFF && r->d[r->pos + 1] == 0xFF) r->pos++;   /* fill */
    if (r->marker) { r->pos += 2; r->marker = 0; r->insufficient = 0; }
    else if (r->pos + 1 < r->n && r->d[r->pos] == 0xFF && r->d[r->pos + 1] >= 0xD0 && r->d[r->pos + 1] <= 0xD7) {
        r->pos += 2; r->insufficient = 0;
    }
    pred[0] = pred[1] = pred[2] = 0; *eobrun = 0;
}

/* jdhuff.c decode_mcu, one block of a sequential scan */
static void seq_block(bitr *r, const dtbl *dc, const dtbl *ac, int16_t *blk, int *pred) {
    int s = decode_sym(r, dc);
    *pred += s ? extend(get_bits(r, s), s) : 0;
    blk[0] = (int16_t)*pred;
    for (int k = 1; k < 64; k++) {
        int rs = decode_sym(r, ac), rr = rs >> 4, ss = rs & 15;
        if (ss) { k += rr; if (k > 63) break; blk[k] = (int16_t)extend(get_bits(r, ss), ss); }
        else { if (rr != 15) break; k += 15; }
    }
}

/* ------------------------------------------------------------------ progressive (SOF2) decode: jdphuff.c
 * What the reference as shipped writes (NVJPEG_ENCODING_PROGRESSIVE_DCT_HUFFMAN, ImageCompressorImpl.cu:28; SURVEY.md
 * 8f N4). All scans are absorbed into the coefficient array (jdapimin.c without buffered-image mode), then the common
 * back end runs: block smoothing never triggers on a complete file. */

/* jdphuff.c start_pass_phuff_decoder: scan parameters libjpeg accepts (a refinement refines by one bit), and coef_bits
 * (the Al of the last scan that sent each of zig-zag 0..9, -1: none yet) */
static int prog_scan_ok(const pscan *sc) {
    return !(sc->Ss > sc->Se || sc->Se > 63 || (sc->Ss == 0 && sc->Se != 0) || (sc->Ss > 0 && sc->ncomp != 1) ||
             sc->Al > 13 || (sc->Ah != 0 && sc->Al != sc->Ah - 1));
}
static void note_coef_bits(int cb[3][10], const pscan *sc) {
    for (int i = 0; i < sc->ncomp; i++)
        for (int k = sc->Ss; k <= sc->Se && k < 10; k++) cb[sc->comp[i]][k] = sc->Al;
}
/* jdcoefct.c smoothing_ok (libjpeg-turbo 2.1 and later): every component's DC sent, the quantisers of zig-zag 0..9
 * non-zero, and some coefficient among zig-zag 1..9 of an output component (0..nout-1) unfinished. libjpeg would then
 * block-smooth the output, which this checker does not restate: -18. */
static int prog_smoothed(const int cb[3][10], int ncomp, int nout, const uint16_t *qt[3]) {
    int unfinished = 0;
    for (int c = 0; c < ncomp; c++) {
        if (cb[c][0] < 0) return 0;
        for (int k = 0; k < 10; k++) if (qt[c][ZIGZAG[k]] == 0) return 0;
        for (int k = 1; k < 10; k++) if (c < nout && cb[c][k] != 0) unfinished = 1;
    }
    return unfinished ? -18 : 0;
}

static void prog_block(bitr *r, const pscan *sc, int ci, const dtbl *dc, const dtbl *ac, int16_t *blk, int *pred, int *eobrun) {
    const int Al = sc->Al, p1 = 1 << Al, m1 = -(1 << Al);
    if (sc->Ss == 0) {
        if (sc->Ah == 0) { /* decode_mcu_DC_first */
            int s = decode_sym(r, dc);
            int diff = s ? extend(get_bits(r, s), s) : 0;
            pred[ci] += diff;
            blk[0] = (int16_t)(pred[ci] * (1 << Al));
        } else {           /* decode_mcu_DC_refine */
            if (get_bit(r)) blk[0] |= (int16_t)p1;
        }
        return;
    }
    if (sc->Ah == 0) {     /* decode_mcu_AC_first */
        if (*eobrun > 0) { (*eobrun)--; return; }
        for (int k = sc->Ss; k <= sc->Se; k++) {
            int rs = decode_sym(r, ac), rr = rs >> 4, ss = rs & 15;
            if (ss) {
                k += rr;
                int v = extend(get_bits(r, ss), ss);
                if (k <= 63) blk[k] = (int16_t)(v * (1 << Al));
            } else {
                if (rr == 15) k += 15;
                else { *eobrun = 1 << rr; if (rr) *eobrun += get_bits(r, rr); (*eobrun)--; break; }
            }
        }
        return;
    }
    /* decode_mcu_AC_refine */
    int k = sc->Ss;
    if (*eobrun == 0) {
        for (; k <= sc->Se; k++) {
            int rs = decode_sym(r, ac), rr = rs >> 4, ss = rs & 15, val = 0;
            if (ss) val = get_bit(r) ? p1 : m1;       /* size of a new coefficient is always 1 */
            else if (rr != 15) { *eobrun = 1 << rr; if (rr) *eobrun += get_bits(r, rr); break; }
            /* advance over already-nonzero coefficients and rr still-zero ones, refining the nonzero ones */
            do {
                int16_t *cp = blk + k;
                if (*cp != 0) {
                    if (get_bit(r) && (*cp & p1) == 0) *cp = (int16_t)(*cp + (*cp >= 0 ? p1 : m1));
                } else {
                    if (--rr < 0) break;
                }
                k++;
            } while (k <= sc->Se);
            if (val && k <= 63) blk[k] = (int16_t)val;
        }
    }
    if (*eobrun > 0) {
        for (; k <= sc->Se; k++) {
            int16_t *cp = blk + k;
            if (*cp != 0 && get_bit(r) && (*cp & p1) == 0) *cp = (int16_t)(*cp + (*cp >= 0 ? p1 : m1));
        }
        (*eobrun)--;
    }
}

/* One scan into the scan-order coefficient array. A sequential scan and an interleaved progressive one run in MCU
 * order over every block of the MCU (padding blocks too), a one-component progressive scan in raster order over the
 * component's own blocks (real data only). In a progressive scan an MCU that starts after the data ran out
 * (insufficient_data) is left alone. dc[i] / ac[i]: the tables of the scan's i-th component. */
static void decode_scan(bitr *r, const orc_geom *g, const pscan *sc, int prog, int ri, const dtbl *dc, const dtbl *ac,
                        int16_t *coef) {
    int pred[3] = {0, 0, 0}, eobrun = 0, togo = ri;
    if (!prog || sc->ncomp > 1) {
        for (long long mi = 0; mi < (long long)g->mcux * g->mcuy; mi++) {
            if (ri && togo == 0) { prog_restart(r, pred, &eobrun); togo = ri; }
            for (int i = 0; i < sc->ncomp && !(prog && r->insufficient); i++) {
                int c = sc->comp[i], nb = c ? 1 : g->hs * g->vs, b0 = c ? g->bpm - 3 + c : 0;
                for (int b = 0; b < nb; b++) {
                    int16_t *blk = coef + ((size_t)mi * g->bpm + b0 + b) * 64;
                    if (prog) prog_block(r, sc, i, &dc[i], &ac[i], blk, pred, &eobrun);
                    else seq_block(r, &dc[i], &ac[i], blk, &pred[i]);
                }
            }
            if (ri) togo--;
        }
    } else {
        int c = sc->comp[0];
        for (int by = 0; by < g->hib[c]; by++)
            for (int bx = 0; bx < g->wib[c]; bx++) {
                if (ri && togo == 0) { prog_restart(r, pred, &eobrun); togo = ri; }
                if (!r->insufficient) prog_block(r, sc, 0, &dc[0], &ac[0], coef + block_index(g, c, bx, by) * 64, pred, &eobrun);
                if (ri) togo--;
            }
    }
}

/* ------------------------------------------------------------------ decoder: the file reader (jdmarker.c) */

/* jdmarker.c get_interesting_appn: JFIF APP0 ("JFIF\0", 14+ bytes) and Adobe APP14 ("Adobe", 12+ bytes, transform in
 * byte 11); jdapimin.c default_decompress_parms then takes three components as RGB (no colour transform, which this
 * checker does not restate: such files are refused) for Adobe transform 0, or without either marker for ids R, G, B. */
static void note_appn(int m, const uint8_t *s, int n, int *jfif, int *adobe) {
    if (m == 0xE0 && n >= 14 && !memcmp(s, "JFIF", 5)) *jfif = 1;
    if (m == 0xEE && n >= 12 && !memcmp(s, "Adobe", 5)) *adobe = s[11];
}
static int rgb_coded(int jfif, int adobe, const int id[3]) {
    if (jfif) return 0;
    if (adobe >= 0) return adobe == 0;
    return id[0] == 'R' && id[1] == 'G' && id[2] == 'B';
}

typedef struct {
    orc_geom g;           /* three components: css 0..4; one: ORC_CSS_GRAY, laid out 1x1 whatever its SOF says */
    int ncomp, sof;       /* 1 or 3; 0xC0 / 0xC1 (sequential) or 0xC2 (progressive) */
    uint16_t qt[3][64];   /* natural order, per component, as the last scan found them */
    int16_t *coef;        /* scan-order blocks of g, zig-zag order (malloc'ed) */
} jfile;

enum { READ_FRAME, READ_HEADERS, READ_ALL };

/* The one marker walker: SOF0/1/2 with one or three components, DQT (8 and 16 bit), DHT, DRI, APP0/APP14 and every SOS.
 * READ_FRAME stops after the SOF (a size query); READ_HEADERS stops at the first SOS of a three-component sequential
 * file and describes it in *info (orc_parse); READ_ALL decodes every scan into f->coef and applies the smoothing rule to
 * output components 0..nout-1. A three-component sequential file is what the product decodes: one interleaved scan,
 * components in SOF order, chroma sharing their tables; nothing after that scan is read. */
static int read_file(const uint8_t *jpg, size_t len, int upto, int nout, jfile *f, orc_info *info) {
    memset(f, 0, sizeof(*f));
    if (len < 4 || jpg[0] != 0xFF || jpg[1] != 0xD8) return -1;
    uint16_t qtabs[4][64]; int have_q[4] = {0, 0, 0, 0};
    uint8_t hb[2][4][17], hv[2][4][256];
    memset(hb, 0, sizeof(hb)); memset(hv, 0, sizeof(hv));
    int id[3] = {-1, -1, -1}, tq[3] = {0, 0, 0}, seq3 = 0, ri = 0, jfif = 0, adobe = -1, nscans = 0, cb[3][10];
    memset(cb, 0xFF, sizeof(cb));
    size_t p = 2;
    int rc = -15;
    while (p + 2 <= len) {
        if (jpg[p] != 0xFF) { rc = -2; break; }
        int m = jpg[p + 1];
        if (m == 0xFF) { p++; continue; }
        p += 2;
        if (m == 0xD8 || (m >= 0xD0 && m <= 0xD7) || m == 0x01) continue;
        if (m == 0xD9) { rc = f->coef && !seq3 ? 0 : -3; break; }
        if (p + 2 > len) { rc = -4; break; }
        int L = rd16(jpg + p);
        if (L < 2 || p + L > len) { rc = -4; break; }
        const uint8_t *s = jpg + p + 2; int n = L - 2;
        if (m == 0xDB) {
            while (n > 0) {
                int pq = s[0] >> 4, t = s[0] & 15; s++; n--;
                if (t > 3) { rc = -5; goto done; }
                for (int k = 0; k < 64; k++) qtabs[t][ZIGZAG[k]] = (uint16_t)(pq ? rd16(s + 2 * k) : s[k]);
                s += pq ? 128 : 64; n -= pq ? 128 : 64; have_q[t] = 1;
            }
        } else if (m == 0xC0 || m == 0xC1 || m == 0xC2) {
            if (f->sof || s[0] != 8) { rc = -6; break; }
            int nc = s[5], H = rd16(s + 1), W = rd16(s + 3), samp[3] = {0, 0, 0}, css = ORC_CSS_GRAY;
            if (nc != 1 && nc != 3) { rc = -7; break; }
            for (int c = 0; c < nc; c++) {
                id[c] = s[6 + 3 * c]; samp[c] = s[7 + 3 * c]; tq[c] = s[8 + 3 * c];
                if (tq[c] > 3) { rc = -14; goto done; }
            }
            if (W <= 0 || H <= 0) { rc = -13; break; }
            if (nc == 3) {
                if (samp[1] != 0x11 || samp[2] != 0x11 || tq[1] != tq[2]) { rc = -11; break; }
                css = css_of(samp[0] >> 4, samp[0] & 15);
                if (css < 0) { rc = -13; break; }
            }
            seq3 = m != 0xC2 && nc == 3;
            if (upto == READ_HEADERS && !seq3) { rc = m == 0xC2 ? -8 : -7; break; }
            f->ncomp = nc; f->sof = m;
            layout(W, H, css, &f->g);
            if (upto == READ_FRAME) return 0;
            if (upto == READ_ALL && !(f->coef = (int16_t *)calloc((size_t)f->g.nblocks * 64, 2))) { rc = -2; break; }
        } else if (m >= 0xC3 && m <= 0xCF && m != 0xC4 && m != 0xC8 && m != 0xCC) {
            rc = -8; break;   /* lossless / arithmetic */
        } else if (m == 0xC4) {
            while (n > 0) {
                int tc = s[0] >> 4, th = s[0] & 15; s++; n--;
                if (tc > 1 || th > 3) { rc = -9; goto done; }
                int ns = 0; hb[tc][th][0] = 0;
                for (int l = 1; l <= 16; l++) { hb[tc][th][l] = s[l - 1]; ns += s[l - 1]; }
                s += 16; n -= 16;
                if (ns > 256) { rc = -9; goto done; }
                memset(hv[tc][th], 0, 256); memcpy(hv[tc][th], s, ns); s += ns; n -= ns;
            }
        } else if (m == 0xDD) {
            ri = rd16(s);
        } else if (m == 0xDA) {
            if (!f->sof) { rc = -10; break; }
            if (nscans++ == 0 && f->ncomp == 3 && rgb_coded(jfif, adobe, id)) { rc = -17; break; }
            pscan sc; memset(&sc, 0, sizeof(sc));
            sc.ncomp = s[0];
            if (sc.ncomp < 1 || sc.ncomp > f->ncomp) { rc = -10; break; }
            for (int i = 0; i < sc.ncomp; i++) {
                sc.comp[i] = -1;
                for (int c = 0; c < f->ncomp; c++) if (id[c] == s[1 + 2 * i]) sc.comp[i] = c;
                sc.td[i] = s[2 + 2 * i] >> 4; sc.ta[i] = s[2 + 2 * i] & 15;
                if (sc.comp[i] < 0 || sc.td[i] > 3 || sc.ta[i] > 3) { rc = -10; goto done; }
            }
            sc.Ss = s[1 + 2 * sc.ncomp]; sc.Se = s[2 + 2 * sc.ncomp];
            sc.Ah = s[3 + 2 * sc.ncomp] >> 4; sc.Al = s[3 + 2 * sc.ncomp] & 15;
            if (seq3) {
                if (sc.ncomp != 3 || sc.comp[0] != 0 || sc.comp[1] != 1 || sc.comp[2] != 2) { rc = -10; break; }
                if (sc.td[1] != sc.td[2] || sc.ta[1] != sc.ta[2]) { rc = -12; break; }
            }
            if (f->sof == 0xC2) {
                if (!prog_scan_ok(&sc)) { rc = -16; break; }
                note_coef_bits(cb, &sc);
            }
            for (int c = 0; c < f->ncomp; c++) {
                if (!have_q[tq[c]]) { rc = -14; goto done; }
                memcpy(f->qt[c], qtabs[tq[c]], 128);
            }
            size_t e0 = p + L, e = entropy_end(jpg, len, e0);
            if (upto == READ_HEADERS) {
                info->W = f->g.W; info->H = f->g.H; info->css = f->g.css; info->hs = f->g.hs; info->vs = f->g.vs;
                info->restart_interval = ri; info->scan_offset = e0; info->scan_len = e - e0;
                memcpy(info->qt, f->qt, sizeof(info->qt));
                for (int t = 0; t < 4; t++) {   /* DC0, AC0, DC1, AC1 */
                    int sel = t & 1 ? sc.ta[t >> 1] : sc.td[t >> 1];
                    memcpy(info->bits[t], hb[t & 1][sel], 17); memcpy(info->vals[t], hv[t & 1][sel], 256);
                }
                return 0;
            }
            bitr r = {jpg + e0, e - e0, 0, 0, 0, 0, 0};
            dtbl dct[3], act[3];
            for (int i = 0; i < sc.ncomp; i++) {
                make_dtbl(hb[0][sc.td[i]], hv[0][sc.td[i]], &dct[i]);
                make_dtbl(hb[1][sc.ta[i]], hv[1][sc.ta[i]], &act[i]);
            }
            decode_scan(&r, &f->g, &sc, f->sof == 0xC2, ri, dct, act, f->coef);
            if (seq3) { rc = 0; break; }
            p = e;
            continue;
        } else {
            note_appn(m, s, n, &jfif, &adobe);
        }
        p += L;
    }
    /* the data ended after a scan without EOI: jdatasrc.c inserts one */
    if (rc == -15 && f->sof == 0xC2 && f->coef && nscans > 0) rc = 0;
    if (rc == 0 && f->sof == 0xC2) {
        const uint16_t *q[3] = {qtabs[tq[0]], qtabs[tq[1]], qtabs[tq[2]]};
        rc = prog_smoothed((const int(*)[10])cb, f->ncomp, nout, q);
    }
done:
    if (rc) { free(f->coef); f->coef = NULL; }
    return rc;
}

int orc_parse(const uint8_t *jpg, size_t len, orc_info *info) {
    jfile f;
    memset(info, 0, sizeof(*info));
    return read_file(jpg, len, READ_HEADERS, 3, &f, info);
}

int orc_decode_coefs(const uint8_t *jpg, size_t len, const orc_info *info, int16_t *coef) {
    orc_geom g; if (orc_geometry(info->W, info->H, info->css, &g)) return -1;
    if (info->scan_offset + info->scan_len > len) return -2;
    dtbl dc[3], ac[3];
    for (int c = 0; c < 3; c++) {
        make_dtbl(info->bits[c ? 2 : 0], info->vals[c ? 2 : 0], &dc[c]);
        make_dtbl(info->bits[c ? 3 : 1], info->vals[c ? 3 : 1], &ac[c]);
    }
    pscan sc = {3, {0, 1, 2}, {0, 0, 0}, {0, 0, 0}, 0, 63, 0, 0};
    bitr r = {jpg + info->scan_offset, info->scan_len, 0, 0, 0, 0, 0};
    memset(coef, 0, (size_t)g.nblocks * 128);
    decode_scan(&r, &g, &sc, 0, info->restart_interval, dc, ac, coef);
    return 0;
}

/* ------------------------------------------------------------------ A.9 back end: IDCT (jidctint.c jpeg_idct_islow,
 * jidctred.c), upsampling (jdsample.c), colour (jdcolor.c) */

static void idct_1d(const int *in, int stride, int *out, int sh) {
    int i0 = in[0], i1 = in[stride], i2 = in[2 * stride], i3 = in[3 * stride], i4 = in[4 * stride],
        i5 = in[5 * stride], i6 = in[6 * stride], i7 = in[7 * stride];
    int z1 = (i2 + i6) * F_0_541;
    int t2 = z1 - i6 * F_1_847, t3 = z1 + i2 * F_0_765;
    int t0 = (i0 + i4) << 13, t1 = (i0 - i4) << 13;
    int t10 = t0 + t3, t13 = t0 - t3, t11 = t1 + t2, t12 = t1 - t2;
    int a0 = i7, a1 = i5, a2 = i3, a3 = i1;
    z1 = a0 + a3; int z2 = a1 + a2, z3 = a0 + a2, z4 = a1 + a3;
    int z5 = (z3 + z4) * F_1_175;
    a0 *= F_0_298; a1 *= F_2_053; a2 *= F_3_072; a3 *= F_1_501;
    z1 *= -F_0_899; z2 *= -F_2_562; z3 = z3 * (-F_1_961) + z5; z4 = z4 * (-F_0_390) + z5;
    a0 += z1 + z3; a1 += z2 + z4; a2 += z2 + z3; a3 += z1 + z4;
    out[0] = DESCALE(t10 + a3, sh); out[7 * stride] = DESCALE(t10 - a3, sh);
    out[stride] = DESCALE(t11 + a2, sh); out[6 * stride] = DESCALE(t11 - a2, sh);
    out[2 * stride] = DESCALE(t12 + a1, sh); out[5 * stride] = DESCALE(t12 - a1, sh);
    out[3 * stride] = DESCALE(t13 + a0, sh); out[4 * stride] = DESCALE(t13 - a0, sh);
}

static void idct_block(const int16_t *zz, const uint16_t *q, uint8_t *dst, int stride) {
    int w[64];
    for (int k = 0; k < 64; k++) w[ZIGZAG[k]] = (int)zz[k] * (int)q[ZIGZAG[k]];
    for (int c = 0; c < 8; c++) idct_1d(w + c, 8, w + c, 11);
    for (int r = 0; r < 8; r++) {
        idct_1d(w + r * 8, 1, w + r * 8, 18);
        for (int c = 0; c < 8; c++) dst[r * stride + c] = (uint8_t)clampi(w[r * 8 + c] + 128, 0, 255);
    }
}

/* k x k samples of one block: jidctint.c's 8 x 8, jidctred.c jpeg_idct_4x4 / 2x2 / 1x1 */
static void idct_scaled(const int16_t *zz, const uint16_t *q, int k, uint8_t *dst, int stride) {
    if (k == 8) { idct_block(zz, q, dst, stride); return; }
    int x[64], ws[64];
    for (int i = 0; i < 64; i++) x[ZIGZAG[i]] = (int)zz[i] * (int)q[ZIGZAG[i]];
    if (k == 1) { dst[0] = (uint8_t)clampi(DESCALE(x[0], 3) + 128, 0, 255); return; }
    if (k == 2) {
        for (int c = 0; c < 8; c++) {   /* columns 2, 4, 6 are never read */
            const int *in = x + c;
            const int t10 = in[0] << 15;
            const int t0 = -5906 * in[56] + 6967 * in[40] - 10426 * in[24] + 29692 * in[8];
            ws[c] = DESCALE(t10 + t0, 13);
            ws[8 + c] = DESCALE(t10 - t0, 13);
        }
        for (int r = 0; r < 2; r++) {
            const int *w = ws + 8 * r;
            const int t10 = w[0] << 15;
            const int t0 = -5906 * w[7] + 6967 * w[5] - 10426 * w[3] + 29692 * w[1];
            dst[r * stride] = (uint8_t)clampi(DESCALE(t10 + t0, 20) + 128, 0, 255);
            dst[r * stride + 1] = (uint8_t)clampi(DESCALE(t10 - t0, 20) + 128, 0, 255);
        }
        return;
    }
    /* k == 4: row / column 4 is never read */
    for (int pass = 0; pass < 2; pass++) {
        const int n = pass ? 4 : 8, sh = pass ? 19 : 12;
        for (int i = 0; i < n; i++) {
            int v[8];
            for (int j = 0; j < 8; j++) v[j] = pass ? ws[i * 8 + j] : x[j * 8 + i];
            const int t0e = v[0] << 14, t2e = 15137 * v[2] - 6270 * v[6];
            const int t10 = t0e + t2e, t12 = t0e - t2e;
            const int z1 = v[7], z2 = v[5], z3 = v[3], z4 = v[1];
            const int t0 = -1730 * z1 + 11893 * z2 - 17799 * z3 + 8697 * z4;
            const int t2 = -4176 * z1 - 4926 * z2 + 7373 * z3 + 20995 * z4;
            const int o[4] = {DESCALE(t10 + t2, sh), DESCALE(t12 + t0, sh), DESCALE(t12 - t0, sh), DESCALE(t10 - t2, sh)};
            for (int j = 0; j < 4; j++) {
                if (pass) dst[i * stride + j] = (uint8_t)clampi(o[j] + 128, 0, 255);
                else ws[j * 8 + i] = o[j];
            }
        }
    }
}

/* jdmaster.c: chroma DCT output size for luma size S */
static int chroma_size(int hs, int vs, int S) {
    int sc = S;
    while (sc < 8 && (hs * S) % (2 * sc) == 0 && (vs * S) % (2 * sc) == 0) sc *= 2;
    return sc;
}

/* jdsample.c: a plane of true size dw x dh (row pitch is) expanded hx x vx into o (row pitch dw * hx). The fancy
 * (triangle) filters run only when the chroma output size is above 1 (do_fancy), h2v1 / h2v2 only on planes wider than
 * 2 samples; everything else is replication (fullsize, int_upsample). */
static void upsample(const uint8_t *in, int is, int dw, int dh, int hx, int vx, int fancy, uint8_t *o) {
    const int ow = dw * hx, oh = dh * vx;
#define IN(r, i) ((int)in[(size_t)(r) * is + (i)])
    if (hx == 2 && vx == 1 && fancy && dw > 2) {          /* h2v1_fancy_upsample */
        for (int r = 0; r < dh; r++) {
            uint8_t *d = o + (size_t)r * ow;
            for (int i = 0; i < dw; i++) {
                d[2 * i] = (uint8_t)(i == 0 ? IN(r, 0) : (3 * IN(r, i) + IN(r, i - 1) + 1) >> 2);
                d[2 * i + 1] = (uint8_t)(i == dw - 1 ? IN(r, dw - 1) : (3 * IN(r, i) + IN(r, i + 1) + 2) >> 2);
            }
        }
    } else if (hx == 1 && vx == 2 && fancy) {             /* h1v2_fancy_upsample */
        for (int r = 0; r < dh; r++) {
            int ra = r > 0 ? r - 1 : 0, rb = r < dh - 1 ? r + 1 : dh - 1;
            for (int i = 0; i < dw; i++) {
                o[(size_t)(2 * r) * ow + i] = (uint8_t)((3 * IN(r, i) + IN(ra, i) + 1) >> 2);
                o[(size_t)(2 * r + 1) * ow + i] = (uint8_t)((3 * IN(r, i) + IN(rb, i) + 2) >> 2);
            }
        }
    } else if (hx == 2 && vx == 2 && fancy && dw > 2) {   /* h2v2_fancy_upsample */
        for (int r = 0; r < dh; r++)
            for (int half = 0; half < 2; half++) {
                int rn = half == 0 ? (r > 0 ? r - 1 : 0) : (r < dh - 1 ? r + 1 : dh - 1);
                uint8_t *d = o + (size_t)(2 * r + half) * ow;
                for (int i = 0; i < dw; i++) {
                    int s = 3 * IN(r, i) + IN(rn, i);
                    int sl = i > 0 ? 3 * IN(r, i - 1) + IN(rn, i - 1) : 0;
                    int sr = i < dw - 1 ? 3 * IN(r, i + 1) + IN(rn, i + 1) : 0;
                    d[2 * i] = (uint8_t)(i == 0 ? (4 * s + 8) >> 4 : (3 * s + sl + 8) >> 4);
                    d[2 * i + 1] = (uint8_t)(i == dw - 1 ? (4 * s + 7) >> 4 : (3 * s + sr + 7) >> 4);
                }
            }
    } else {
        for (int r = 0; r < oh; r++)
            for (int i = 0; i < ow; i++) o[(size_t)r * ow + i] = (uint8_t)IN(r / vx, i / hx);
    }
#undef IN
}

/* Coefficients -> what libjpeg returns with scale_denom 8 / S (jdmaster.c): ceil(W S / 8) x ceil(H S / 8) gray samples
 * (luma only: no chroma IDCT, no upsampling, no colour conversion) or BGR. Luma blocks come out S x S, chroma blocks at
 * chroma_size's size, the chroma planes at their true size ceil(W Sc / (hs 8)) x ceil(H Sc / (vs 8)). */
static int render(const orc_geom *g, const uint16_t qt[3][64], const int16_t *coef, int S, int gray, uint8_t *out,
                  size_t step) {
    const int nc = gray ? 1 : 3, Sc = chroma_size(g->hs, g->vs, S);
    const int Wo = ceil_div(g->W * S, 8), Ho = ceil_div(g->H * S, 8);
    const int hx = g->hs * S / Sc, vx = g->vs * S / Sc;
    const int dw = ceil_div(g->W * Sc, g->hs * 8), dh = ceil_div(g->H * Sc, g->vs * 8), ow = dw * hx;
    uint8_t *pl[3] = {NULL, NULL, NULL}, *up[3] = {NULL, NULL, NULL};
    int pw[3], k[3], rc = 0;
    for (int c = 0; c < nc; c++) {
        int h = c ? 1 : g->hs, v = c ? 1 : g->vs;
        k[c] = c ? Sc : S;
        pw[c] = g->mcux * h * k[c];
        pl[c] = (uint8_t *)malloc((size_t)pw[c] * g->mcuy * v * k[c]);
        if (c) up[c] = (uint8_t *)malloc((size_t)ow * dh * vx);
        if (!pl[c] || (c && !up[c])) { rc = -2; goto done; }
    }
    for (int my = 0; my < g->mcuy; my++)
        for (int mx = 0; mx < g->mcux; mx++) {
            const int16_t *mcu = coef + ((size_t)my * g->mcux + mx) * g->bpm * 64;
            int blkn = 0;
            for (int c = 0; c < nc; c++) {
                int h = c ? 1 : g->hs, v = c ? 1 : g->vs;
                for (int by = 0; by < v; by++)
                    for (int bx = 0; bx < h; bx++, blkn++)
                        idct_scaled(mcu + blkn * 64, qt[c], k[c],
                                   pl[c] + (size_t)(my * v + by) * k[c] * pw[c] + (size_t)(mx * h + bx) * k[c], pw[c]);
            }
        }
    if (gray) {
        for (int y = 0; y < Ho; y++) memcpy(out + (size_t)y * step, pl[0] + (size_t)y * pw[0], (size_t)Wo);
        goto done;
    }
    for (int c = 1; c < 3; c++) upsample(pl[c], pw[c], dw, dh, hx, vx, Sc > 1, up[c]);
    for (int y = 0; y < Ho; y++)   /* jdcolor.c ycc_rgb_convert */
        for (int x = 0; x < Wo; x++) {
            int Y = pl[0][(size_t)y * pw[0] + x];
            int cb = up[1][(size_t)y * ow + x] - 128, cr = up[2][(size_t)y * ow + x] - 128;
            int r = Y + ((91881 * cr + 32768) >> 16);
            int b = Y + ((116130 * cb + 32768) >> 16);
            int gg = Y + ((-22554 * cb - 46802 * cr + 32768) >> 16);
            uint8_t *p = out + (size_t)y * step + (size_t)x * 3;
            p[0] = (uint8_t)clampi(b, 0, 255); p[1] = (uint8_t)clampi(gg, 0, 255); p[2] = (uint8_t)clampi(r, 0, 255);
        }
done:
    for (int c = 0; c < 3; c++) { free(pl[c]); free(up[c]); }
    return rc;
}

int orc_inverse(const int16_t *coef, const orc_info *info, uint8_t *bgr, size_t step) {
    orc_geom g; if (orc_geometry(info->W, info->H, info->css, &g)) return -1;
    uint16_t qt[3][64];
    memcpy(qt[0], info->qt[0], 128); memcpy(qt[1], info->qt[1], 128); memcpy(qt[2], info->qt[1], 128);
    return render(&g, (const uint16_t(*)[64])qt, coef, 8, 0, bgr, step);
}

/* ------------------------------------------------------------------ decoder: entry points */

int orc_decode_output(const uint8_t *jpg, size_t len, int denom, int gray_out, uint8_t *out, size_t step, int *W, int *H) {
    if (denom != 1 && denom != 2 && denom != 4 && denom != 8) return -20;
    jfile f;
    int rc = read_file(jpg, len, out ? READ_ALL : READ_FRAME, gray_out ? 1 : 3, &f, NULL);
    if (rc) return rc;
    if (!gray_out && f.ncomp == 1) rc = -21;
    else {
        if (W) *W = ceil_div(f.g.W, denom);
        if (H) *H = ceil_div(f.g.H, denom);
        if (out) rc = render(&f.g, (const uint16_t(*)[64])f.qt, f.coef, 8 / denom, gray_out, out, step);
    }
    free(f.coef);
    return rc;
}

int orc_decode(const uint8_t *jpg, size_t len, uint8_t *bgr, size_t step, int *W, int *H) {
    return orc_decode_output(jpg, len, 1, 0, bgr, step, W, H);
}

int orc_decode_progressive(const uint8_t *jpg, size_t len, uint8_t *bgr, size_t step, int *W, int *H) {
    jfile f;
    int rc = read_file(jpg, len, READ_FRAME, 3, &f, NULL);
    if (!rc && f.sof != 0xC2) rc = -8;
    return rc ? rc : orc_decode(jpg, len, bgr, step, W, H);
}

/* ------------------------------------------------------------------ a-12: difference map + PSNR */

void orc_diff(const uint8_t *a, const uint8_t *b, size_t n, int mode, uint8_t *out) {
    for (size_t i = 0; i < n; i++) {
        int d = (int)a[i] - (int)b[i];
        out[i] = (uint8_t)(mode == 0 ? (d < 0 ? -d : d) : clampi(d + 128, 0, 255));
    }
}
uint64_t orc_ssd(const uint8_t *a, const uint8_t *b, size_t n) {
    uint64_t s = 0;
    for (size_t i = 0; i < n; i++) { int d = (int)a[i] - (int)b[i]; s += (uint64_t)(d * d); }
    return s;
}
double orc_psnr(const uint8_t *a, const uint8_t *b, size_t n) {
    uint64_t s = orc_ssd(a, b, n);
    /* cv::PSNR: 20*log10(255/(sqrt(ssd/n)+DBL_EPSILON)) */
    double diff = sqrt((double)s / (double)n);
    return 20.0 * log10(255.0 / (diff + 2.220446049250313e-16));
}
