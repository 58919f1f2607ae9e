/*
 * gray_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE: the grayscale (one-component, JCS_GRAYSCALE) half of the CPU
 * checker. It includes oracle/jpeg_oracle.c and reuses its libjpeg-turbo restatement unchanged (islow FDCT / IDCT,
 * quantiser, symbol statistics, jpeg_gen_optimal_table, entropy coder, stuffing, Huffman decoding, the progressive
 * block decoder), adding only what a one-component stream does differently:
 *   encode: the samples are Y as they stand (jccolor.c grayscale_convert), edges replicated to whole blocks
 *           (jcsample.c expand_right_edge, jcprepct.c), quantised with the luma table; DC0/AC0 only; one DQT, SOF0 and
 *           SOS with one component; the restart interval counts blocks (a one-component scan is non-interleaved: one
 *           block per MCU);
 *   decode: a one-component file (baseline or progressive, any sampling factor in its SOF: its scans are
 *           non-interleaved, laid out 1x1) or the Y plane of a three-component file -- what libjpeg returns with
 *           out_color_space = JCS_GRAYSCALE: no chroma IDCT, no upsampling, no colour conversion.
 * tests/gray_oracle.py compiles it (gcc, into a temporary directory) and binds it; tests/test_oracle_gray.py pins it
 * to cv2 (libjpeg-turbo 3.1.2) and to tests/golden/golden_gray.json.
 */
#include "../../oracle/jpeg_oracle.c"

#define GRAY_CSS 6   /* B2J_CSS_GRAY */

static void gray_geometry(int W, int H, orc_geom *g) {
    memset(g, 0, sizeof(*g));
    g->W = W; g->H = H; g->css = GRAY_CSS; g->hs = g->vs = 1;
    g->mcux = ceil_div(W, 8); g->mcuy = ceil_div(H, 8); g->bpm = 1;
    g->dw[0] = W; g->dh[0] = H; g->wib[0] = g->mcux; g->hib[0] = g->mcuy;
    g->nblocks = (long long)g->mcux * g->mcuy;
}

/* jcmarker.c for one component: SOI, JFIF APP0, DQT 0, SOF0 (id 1, 1x1, Tq 0), DHT DC0 + AC0, DRI if set, SOS */
static size_t gray_headers(int W, int H, const uint16_t qt[64], const uint8_t *dc_bits, const uint8_t *dc_vals,
                           const uint8_t *ac_bits, const uint8_t *ac_vals, int restart_interval, uint8_t *out, size_t cap) {
    uint8_t buf[1024]; size_t n = 0;
#define PUT(b) buf[n++] = (uint8_t)(b)
    PUT(0xFF); PUT(0xD8);
    PUT(0xFF); PUT(0xE0); PUT(0); PUT(16); PUT('J'); PUT('F'); PUT('I'); PUT('F'); PUT(0); PUT(1); PUT(1); PUT(0);
    PUT(0); PUT(1); PUT(0); PUT(1); PUT(0); PUT(0);
    PUT(0xFF); PUT(0xDB); PUT(0); PUT(67); PUT(0);
    for (int k = 0; k < 64; k++) PUT(qt[ZIGZAG[k]]);
    PUT(0xFF); PUT(0xC0); PUT(0); PUT(11); PUT(8); PUT(H >> 8); PUT(H & 255); PUT(W >> 8); PUT(W & 255); PUT(1);
    PUT(1); PUT(0x11); PUT(0);
    for (int t = 0; t < 2; t++) {
        const uint8_t *bits = t ? ac_bits : dc_bits, *vals = t ? ac_vals : dc_vals;
        int ns = 0; for (int l = 1; l <= 16; l++) ns += bits[l];
        PUT(0xFF); PUT(0xC4); PUT((19 + ns) >> 8); PUT((19 + ns) & 255); PUT(t ? 0x10 : 0x00);
        for (int l = 1; l <= 16; l++) PUT(bits[l]);
        for (int i = 0; i < ns; i++) PUT(vals[i]);
    }
    if (restart_interval) { PUT(0xFF); PUT(0xDD); PUT(0); PUT(4); PUT(restart_interval >> 8); PUT(restart_interval & 255); }
    PUT(0xFF); PUT(0xDA); PUT(0); PUT(8); PUT(1); PUT(1); PUT(0x00); PUT(0); PUT(63); PUT(0);
#undef PUT
    if (n > cap) return 0;
    memcpy(out, buf, n);
    return n;
}

/* 8-bit samples with row pitch `step` -> the stream libjpeg-turbo writes; restart interval in blocks (0 = none) */
int orc_encode_gray(const uint8_t *gray, size_t step, int W, int H, int quality, int optimize, int ri, uint8_t *out,
                    size_t cap, size_t *len) {
    if (W <= 0 || H <= 0 || W > 65535 || H > 65535 || ri < 0 || ri > 65535) return -1;
    orc_geom g; gray_geometry(W, H, &g);
    uint16_t qt[2][64]; orc_quant_tables(quality, qt);
    int16_t *coef = (int16_t *)malloc((size_t)g.nblocks * 128);
    if (!coef) return -2;
    int nat[64]; uint8_t blk8[64];
    for (int by = 0; by < g.mcuy; by++)
        for (int bx = 0; bx < g.mcux; bx++) {
            for (int r = 0; r < 8; r++)
                for (int c = 0; c < 8; c++) {
                    const int y = by * 8 + r, x = bx * 8 + c;
                    blk8[r * 8 + c] = gray[(size_t)(y < H ? y : H - 1) * step + (x < W ? x : W - 1)];
                }
            fdct_block(blk8, 8, nat);
            int16_t *blk = coef + ((size_t)by * g.mcux + bx) * 64;
            for (int k = 0; k < 64; k++) blk[k] = quantise(nat[ZIGZAG[k]], qt[0][ZIGZAG[k]]);
        }
    /* orc_histogram / orc_entropy_bits with bpm = 1 treat every block as the third component (comp_of_block): one DC
     * predictor and one table pair, in slots [2] / [3] of their arrays -- here the stream's DC0 / AC0 */
    const long long nblk = g.nblocks, iv = ri ? ri : nblk;
    uint8_t bits[4][17], vals[4][256];
    memset(bits, 0, sizeof(bits)); memset(vals, 0, sizeof(vals));
    int rc = 0;
    if (optimize) {
        uint32_t hist[4][257], h1[4][257];
        memset(hist, 0, sizeof(hist));
        for (long long b0 = 0; b0 < nblk; b0 += iv) {   /* predictors restart with every interval (jchuff.c) */
            orc_histogram(coef + b0 * 64, nblk - b0 < iv ? nblk - b0 : iv, 1, NULL, h1);
            for (int t = 2; t < 4; t++) for (int i = 0; i < 257; i++) hist[t][i] += h1[t][i];
        }
        for (int t = 2; t < 4; t++) if (orc_gen_optimal_table(hist[t], bits[t], vals[t]) < 0) rc = -3;
    } else {
        orc_std_table(0, bits[2], vals[2]);
        orc_std_table(1, bits[3], vals[3]);
    }
    size_t o = 0;
    if (!rc) { o = gray_headers(W, H, qt[0], bits[2], vals[2], bits[3], vals[3], ri, out, cap); if (!o) rc = -4; }
    const size_t raw_cap = (size_t)iv * 208 + 16;
    uint8_t *raw = rc ? NULL : (uint8_t *)malloc(raw_cap);
    if (!rc && !raw) rc = -2;
    int rstn = 0;
    for (long long b0 = 0; !rc && b0 < nblk; b0 += iv) {
        uint64_t nbits = 0;
        if (orc_entropy_bits(coef + b0 * 64, nblk - b0 < iv ? nblk - b0 : iv, 1, NULL, (const uint8_t(*)[17])bits,
                             (const uint8_t(*)[256])vals, raw, raw_cap, &nbits)) { rc = -5; break; }
        o += orc_stuff(raw, nbits, out + o, cap > o ? cap - o : 0);
        if (o + 2 > cap) { rc = -6; break; }
        if (b0 + iv < nblk) { out[o++] = 0xFF; out[o++] = (uint8_t)(0xD0 + rstn); rstn = (rstn + 1) & 7; }
    }
    free(coef); free(raw);
    if (rc) return rc;
    if (o + 2 > cap) return -6;
    out[o++] = 0xFF; out[o++] = 0xD9;
    *len = o;
    return 0;
}

static size_t scan_end(const uint8_t *jpg, size_t len, size_t e) {   /* first marker that is not RSTn / stuffed zero */
    while (e + 1 < len) {
        if (jpg[e] == 0xFF && jpg[e + 1] != 0x00 && !(jpg[e + 1] >= 0xD0 && jpg[e + 1] <= 0xD7)) break;
        e++;
    }
    return e + 1 >= len ? len : e;
}

/* Coefficients of the files orc_parse / orc_decode_progressive reject for having one component, and of progressive
 * three-component files: SOF0 / SOF1 with one component, SOF2 with one or three (chroma 1x1). *coef_out: scan-order
 * blocks of *g (malloc'ed; NULL when want == 0), qt_out: the luma (component 0) quantisation table. */
static int other_coefs(const uint8_t *jpg, size_t len, int want, orc_geom *g, uint16_t qt_out[64], int16_t **coef_out) {
    *coef_out = NULL;
    if (len < 4 || jpg[0] != 0xFF || jpg[1] != 0xD8) return -1;
    uint16_t qtabs[4][64]; int have_q[4] = {0, 0, 0, 0};
    static uint8_t hb[2][4][17], hv[2][4][256];
    memset(hb, 0, sizeof(hb)); memset(hv, 0, sizeof(hv));
    int comp_id[3] = {-1, -1, -1}, comp_hv[3] = {0, 0, 0}, comp_tq[3] = {0, 0, 0}, ncomp = 0, ri = 0, sof = 0;
    int16_t *coef = NULL;
    size_t p = 2;
    int rc = -15;
    while (p + 2 <= len) {
        if (jpg[p] != 0xFF) { rc = -2; break; }
        const int m = jpg[p + 1];
        if (m == 0xFF) { p++; continue; }
        p += 2;
        if (m == 0xD8 || (m >= 0xD0 && m <= 0xD7) || m == 0x01) continue;
        if (m == 0xD9) { rc = sof && (coef || !want) ? 0 : -3; break; }
        if (p + 2 > len) { rc = -4; break; }
        const int L = rd16(jpg + p);
        if (L < 2 || p + L > len) { rc = -4; break; }
        const uint8_t *s = jpg + p + 2; int n = L - 2;
        if (m == 0xDB) {
            while (n > 0) {
                const int pq = s[0] >> 4, tq = s[0] & 15; s++; n--;
                if (tq > 3) { rc = -5; goto done; }
                for (int k = 0; k < 64; k++) qtabs[tq][ZIGZAG[k]] = (uint16_t)(pq ? rd16(s + 2 * k) : s[k]);
                s += pq ? 128 : 64; n -= pq ? 128 : 64; have_q[tq] = 1;
            }
        } else if (m == 0xC0 || m == 0xC1 || m == 0xC2) {
            if (sof || s[0] != 8) { rc = -6; break; }
            ncomp = s[5];
            if (ncomp != 1 && !(ncomp == 3 && m == 0xC2)) { rc = -7; break; }
            const int H = rd16(s + 1), W = rd16(s + 3);
            for (int c = 0; c < ncomp; c++) { comp_id[c] = s[6 + 3 * c]; comp_hv[c] = s[7 + 3 * c]; comp_tq[c] = s[8 + 3 * c] & 3; }
            if (W <= 0 || H <= 0) { rc = -13; break; }
            if (ncomp == 1) {
                gray_geometry(W, H, g);
            } else {
                if (comp_hv[1] != 0x11 || comp_hv[2] != 0x11 || comp_tq[1] != comp_tq[2]) { rc = -11; break; }
                static const int HS[5] = {1, 2, 1, 2, 4}, VS[5] = {1, 1, 2, 2, 1};
                int css = -1;
                for (int i = 0; i < 5; i++) if (HS[i] == comp_hv[0] >> 4 && VS[i] == (comp_hv[0] & 15)) css = i;
                if (css < 0 || orc_geometry(W, H, css, g)) { rc = -13; break; }
            }
            sof = m;
            if (!want) { rc = 0; break; }
            coef = (int16_t *)calloc((size_t)g->nblocks * 64, 2);
            if (!coef) { rc = -2; break; }
        } else if (m >= 0xC3 && m <= 0xCF && m != 0xC4 && m != 0xC8 && m != 0xCC) {
            rc = -8; break;   /* lossless / arithmetic */
        } else if (m == 0xC4) {
            while (n > 0) {
                const int tc = s[0] >> 4, th = s[0] & 15; s++; n--;
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
            if (!sof) { rc = -10; break; }
            pscan sc; sc.ncomp = s[0];
            if (sc.ncomp < 1 || sc.ncomp > ncomp) { rc = -10; break; }
            for (int i = 0; i < sc.ncomp; i++) {
                const int id = s[1 + 2 * i]; sc.comp[i] = -1;
                for (int c = 0; c < ncomp; c++) if (comp_id[c] == id) sc.comp[i] = c;
                if (sc.comp[i] < 0) { rc = -10; goto done; }
                sc.td[i] = s[2 + 2 * i] >> 4; sc.ta[i] = s[2 + 2 * i] & 15;
                if (sc.td[i] > 3 || sc.ta[i] > 3) { rc = -10; goto done; }
            }
            sc.Ss = s[1 + 2 * sc.ncomp]; sc.Se = s[2 + 2 * sc.ncomp];
            sc.Ah = s[3 + 2 * sc.ncomp] >> 4; sc.Al = s[3 + 2 * sc.ncomp] & 15;
            if (!have_q[comp_tq[0]]) { rc = -14; break; }
            memcpy(qt_out, qtabs[comp_tq[0]], 128);
            const size_t e0 = p + L, e = scan_end(jpg, len, e0);
            bitr r = {jpg + e0, e - e0, 0, 0, 0, 0};
            dtbl dct[3], act[3];
            for (int i = 0; i < sc.ncomp; i++) {
                make_dtbl(hb[0][sc.td[i]], hv[0][sc.td[i]], &dct[i]);
                make_dtbl(hb[1][sc.ta[i]], hv[1][sc.ta[i]], &act[i]);
            }
            int pred[3] = {0, 0, 0}, eobrun = 0, togo = ri;
            if (sof != 0xC2) {             /* baseline, one component: every block in raster order, DC + AC */
                for (long long b = 0; b < g->nblocks; b++) {
                    if (ri && togo == 0) { prog_restart(&r, pred, &eobrun); togo = ri; }
                    int16_t *blk = coef + b * 64;
                    const int sz = decode_sym(&r, &dct[0]);
                    pred[0] += sz ? extend(get_bits(&r, sz), sz) : 0;
                    blk[0] = (int16_t)pred[0];
                    for (int k = 1; k < 64; k++) {
                        const int rs = decode_sym(&r, &act[0]), rr = rs >> 4, ss = rs & 15;
                        if (ss) { k += rr; if (k > 63) break; blk[k] = (int16_t)extend(get_bits(&r, ss), ss); }
                        else { if (rr != 15) break; k += 15; }
                    }
                    if (ri) togo--;
                }
            } else {
                if (sc.Ss > sc.Se || sc.Se > 63 || (sc.Ss == 0 && sc.Se != 0) || (sc.Ss > 0 && sc.ncomp != 1)) { rc = -16; break; }
                if (sc.ncomp > 1) {        /* interleaved (three components): MCU order, every block of the MCU */
                    for (long long mi = 0; mi < (long long)g->mcux * g->mcuy; mi++) {
                        if (ri && togo == 0) { prog_restart(&r, pred, &eobrun); togo = ri; }
                        for (int i = 0; i < sc.ncomp; i++) {
                            const int c = sc.comp[i], nb = c ? 1 : g->hs * g->vs, b0 = c ? g->bpm - 3 + c : 0;
                            for (int b = 0; b < nb; b++)
                                prog_block(&r, &sc, i, &dct[i], &act[i], coef + ((size_t)mi * g->bpm + b0 + b) * 64, pred, &eobrun);
                        }
                        if (ri) togo--;
                    }
                } else {                   /* one component: raster order over its own blocks */
                    const int c = sc.comp[0];
                    for (int by = 0; by < g->hib[c]; by++)
                        for (int bx = 0; bx < g->wib[c]; bx++) {
                            if (ri && togo == 0) { prog_restart(&r, pred, &eobrun); togo = ri; }
                            prog_block(&r, &sc, 0, &dct[0], &act[0], coef + block_index(g, c, bx, by) * 64, pred, &eobrun);
                            if (ri) togo--;
                        }
                }
            }
            p = e;
            continue;
        }
        p += L;
    }
done:
    if (rc == 0) *coef_out = coef;
    else free(coef);
    return rc;
}

/* gray: (H, W) samples with row pitch `step`, or NULL to query the size */
int orc_decode_gray(const uint8_t *jpg, size_t len, uint8_t *gray, size_t step, int *W, int *H) {
    orc_info info; orc_geom g; uint16_t qt[64]; int16_t *coef = NULL;
    int rc = orc_parse(jpg, len, &info);
    if (rc == 0) {   /* baseline, three components */
        if (orc_geometry(info.W, info.H, info.css, &g)) return -1;
        memcpy(qt, info.qt[0], sizeof(qt));
        if (gray) {
            coef = (int16_t *)malloc((size_t)g.nblocks * 128);
            if (!coef) return -2;
            rc = orc_decode_coefs(jpg, len, &info, coef);
            if (rc) { free(coef); return rc; }
        }
    } else {
        rc = other_coefs(jpg, len, gray != NULL, &g, qt, &coef);
        if (rc) return rc;
    }
    if (W) *W = g.W;
    if (H) *H = g.H;
    if (!gray) return 0;
    const int pw = g.mcux * g.hs * 8, ph = g.mcuy * g.vs * 8;
    uint8_t *pl = (uint8_t *)malloc((size_t)pw * ph);
    if (!pl) { free(coef); return -2; }
    for (int my = 0; my < g.mcuy; my++)   /* the luma blocks of every MCU: the first hs * vs */
        for (int mx = 0; mx < g.mcux; mx++)
            for (int by = 0; by < g.vs; by++)
                for (int bx = 0; bx < g.hs; bx++)
                    idct_block(coef + (((size_t)my * g.mcux + mx) * g.bpm + by * g.hs + bx) * 64, qt,
                               pl + (size_t)(my * g.vs + by) * 8 * pw + (size_t)(mx * g.hs + bx) * 8, pw);
    for (int y = 0; y < g.H; y++) memcpy(gray + (size_t)y * step, pl + (size_t)y * pw, (size_t)g.W);
    free(pl); free(coef);
    return 0;
}
