/*
 * scaled_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE: the reduced-size (DCT-scaled) decode of the CPU checker,
 * what libjpeg-turbo 3.1.2 returns with scale_num = 1, scale_denom = d (d = 1, 2, 4, 8; cv2 IMREAD_REDUCED_*_d).
 * It includes tests/cpp/gray_oracle.c (and through it oracle/jpeg_oracle.c) and reuses their coefficient decoders
 * unchanged: orc_decode_coefs for baseline three-component files (restart markers included) and the gray checker's
 * decoder for one-component files and for progressive files' luma. It restates only the scaled back end:
 *   jdmaster.c  output size ceil(W / d) x ceil(H / d); every component's DCT output size: luma S = 8 / d, chroma starts
 *               at S and doubles while it is below 8 and both (hs S) % (2 Sc) == 0 and (vs S) % (2 Sc) == 0; true
 *               component sizes ceil(W h k / (hs 8)) x ceil(H v k / (vs 8));
 *   jidctred.c  jpeg_idct_1x1 / 2x2 / 4x4 (jidctint.c jpeg_idct_islow for 8x8);
 *   jdsample.c  fancy filters only when the chroma output size is above 1 (do_fancy), else plain replication;
 *   jdcolor.c   unchanged.
 * Progressive three-component files are decoded in gray only (the gray checker keeps the luma table alone); their
 * colour output is pinned by golden digests. tests/scaled_oracle.py compiles and binds it.
 */
#include "gray_oracle.c"

/* jidctred.c: k x k samples of one block (k = 1, 2, 4) or jidctint.c's 8 x 8 */
static void idct_scaled_block(const int16_t *zz, const uint16_t *q, int k, uint8_t *dst, int stride) {
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
static int chroma_scaled(int hs, int vs, int S) {
    int sc = S;
    while (sc < 8 && (hs * S) % (2 * sc) == 0 && (vs * S) % (2 * sc) == 0) sc *= 2;
    return sc;
}

/* out: (H', W', 3) BGR (gray_out = 0) or (H', W') samples (gray_out = 1) with row pitch `step`, or NULL to query the
 * output size. 0 on success; -20 for a scale other than 1, 2, 4, 8; -21 for colour output of a one-component or a
 * progressive file at a reduced scale. denom 1 is the full-size decode (orc_decode / orc_decode_gray). */
int orc_decode_scaled(const uint8_t *jpg, size_t len, int denom, int gray_out, uint8_t *out, size_t step, int *W, int *H) {
    if (denom != 1 && denom != 2 && denom != 4 && denom != 8) return -20;
    if (denom == 1) return gray_out ? orc_decode_gray(jpg, len, out, step, W, H) : orc_decode(jpg, len, out, step, W, H);
    orc_info info; orc_geom g; uint16_t qt[2][64]; int16_t *coef = NULL;
    int rc = orc_parse(jpg, len, &info);
    if (rc == 0) {   /* baseline, three components */
        if (orc_geometry(info.W, info.H, info.css, &g)) return -1;
        memcpy(qt, info.qt, sizeof(qt));
        if (out) {
            coef = (int16_t *)malloc((size_t)g.nblocks * 128);
            if (!coef) return -2;
            rc = orc_decode_coefs(jpg, len, &info, coef);
            if (rc) { free(coef); return rc; }
        }
    } else {
        rc = other_coefs(jpg, len, out != NULL, &g, qt[0], &coef);
        if (rc) return rc;
        if (!gray_out) { free(coef); return -21; }
    }
    const int S = 8 / denom, Wo = ceil_div(g.W * S, 8), Ho = ceil_div(g.H * S, 8);
    if (W) *W = Wo;
    if (H) *H = Ho;
    if (!out) return 0;
    const int nc = gray_out ? 1 : 3, Sc = chroma_scaled(g.hs, g.vs, S);
    uint8_t *pl[3] = {NULL, NULL, NULL};
    int pw[3], ph[3], k[3];
    for (int c = 0; c < nc; c++) {
        const int h = c ? 1 : g.hs, v = c ? 1 : g.vs;
        k[c] = c ? Sc : S;
        pw[c] = g.mcux * h * k[c]; ph[c] = g.mcuy * v * k[c];
        pl[c] = (uint8_t *)malloc((size_t)pw[c] * ph[c]);
        if (!pl[c]) { rc = -2; goto done; }
    }
    for (int my = 0; my < g.mcuy; my++)
        for (int mx = 0; mx < g.mcux; mx++) {
            const int16_t *mcu = coef + ((size_t)my * g.mcux + mx) * g.bpm * 64;
            int blkn = 0;
            for (int c = 0; c < nc; c++) {
                const int h = c ? 1 : g.hs, v = c ? 1 : g.vs;
                for (int by = 0; by < v; by++)
                    for (int bx = 0; bx < h; bx++, blkn++)
                        idct_scaled_block(mcu + blkn * 64, qt[c ? 1 : 0], k[c],
                                          pl[c] + (size_t)(my * v + by) * k[c] * pw[c] + (size_t)(mx * h + bx) * k[c], pw[c]);
            }
        }
    if (gray_out) {
        for (int y = 0; y < Ho; y++) memcpy(out + (size_t)y * step, pl[0] + (size_t)y * pw[0], (size_t)Wo);
        goto done;
    }
    {
        /* chroma to output resolution: expansion hx x vx over the true component size dw x dh */
        const int hx = g.hs * S / Sc, vx = g.vs * S / Sc;
        const int dw = ceil_div(g.W * Sc, g.hs * 8), dh = ceil_div(g.H * Sc, g.vs * 8);
        const int fancy = Sc > 1;
        const int ow = dw * hx, oh = dh * vx;
        uint8_t *up[3] = {NULL, NULL, NULL};
        for (int c = 1; c < 3 && !rc; c++) {
            const uint8_t *in = pl[c]; const int is = pw[c];
            uint8_t *o = (uint8_t *)malloc((size_t)ow * oh);
            if (!o) { rc = -2; break; }
            up[c] = o;
#define IN(r, i) ((int)in[(size_t)(r) * is + (i)])
            if (hx == 2 && vx == 1 && fancy && dw > 2) {   /* h2v1_fancy_upsample */
                for (int r = 0; r < dh; r++) {
                    uint8_t *d = o + (size_t)r * ow;
                    for (int i = 0; i < dw; i++) {
                        d[2 * i] = (uint8_t)(i == 0 ? IN(r, 0) : (3 * IN(r, i) + IN(r, i - 1) + 1) >> 2);
                        d[2 * i + 1] = (uint8_t)(i == dw - 1 ? IN(r, dw - 1) : (3 * IN(r, i) + IN(r, i + 1) + 2) >> 2);
                    }
                }
            } else if (hx == 1 && vx == 2 && fancy) {        /* h1v2_fancy_upsample */
                for (int r = 0; r < dh; r++) {
                    const int ra = r > 0 ? r - 1 : 0, rb = r < dh - 1 ? r + 1 : dh - 1;
                    for (int i = 0; i < dw; i++) {
                        o[(size_t)(2 * r) * ow + i] = (uint8_t)((3 * IN(r, i) + IN(ra, i) + 1) >> 2);
                        o[(size_t)(2 * r + 1) * ow + i] = (uint8_t)((3 * IN(r, i) + IN(rb, i) + 2) >> 2);
                    }
                }
            } else {                                         /* fullsize / h2v1 / int_upsample: replication */
                for (int r = 0; r < oh; r++)
                    for (int i = 0; i < ow; i++) o[(size_t)r * ow + i] = (uint8_t)IN(r / vx, i / hx);
            }
#undef IN
        }
        if (!rc)
            for (int y = 0; y < Ho; y++)
                for (int x = 0; x < Wo; x++) {
                    const int Y = pl[0][(size_t)y * pw[0] + x];
                    const int cb = up[1][(size_t)y * ow + x] - 128, cr = up[2][(size_t)y * ow + x] - 128;
                    const int r = Y + ((91881 * cr + 32768) >> 16);
                    const int b = Y + ((116130 * cb + 32768) >> 16);
                    const int gg = Y + ((-22554 * cb - 46802 * cr + 32768) >> 16);
                    uint8_t *p = out + (size_t)y * step + (size_t)x * 3;
                    p[0] = (uint8_t)clampi(b, 0, 255); p[1] = (uint8_t)clampi(gg, 0, 255); p[2] = (uint8_t)clampi(r, 0, 255);
                }
        free(up[1]); free(up[2]);
    }
done:
    for (int c = 0; c < 3; c++) free(pl[c]);
    free(coef);
    return rc;
}
