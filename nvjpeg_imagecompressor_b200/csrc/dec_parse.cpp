// dec_parse.cpp -- host-side marker parser (the reference does this with nvjpegGetImageInfo + nvjpegJpegStreamParse,
// ImageCompressorImpl.cu:335,362; semantics follow libjpeg jdmarker.c for the baseline subset listed in dec.h).
#include <stdlib.h>
#include <string.h>

#include <new>

#include "dec.h"
#include "dec_kernels.h"

namespace b2j {

static inline int be16(const uint8_t *p) { return (p[0] << 8) | p[1]; }

// The colour-space markers, as jdmarker.c get_interesting_appn reads them: a JFIF APP0 ("JFIF\0", at least 14 bytes)
// and an Adobe APP14 ("Adobe", at least 12 bytes, the transform in byte 11; the last one seen counts).
struct ColourMarkers {
    bool jfif = false;
    int adobe = -1;   // the Adobe transform, -1: no Adobe marker
    void note(int m, const uint8_t *s, int n) {
        if (m == 0xE0 && n >= 14 && !memcmp(s, "JFIF", 5)) jfif = true;
        if (m == 0xEE && n >= 12 && !memcmp(s, "Adobe", 5)) adobe = s[11];
    }
    // jdapimin.c default_decompress_parms for three components: JFIF means YCbCr; else an Adobe marker decides
    // (transform 0: RGB); else the component ids 'R', 'G', 'B' mean RGB; anything else is YCbCr. RGB-coded files
    // have no colour transform, which the back end always applies, so they are refused.
    bool rgb(const int cid[3]) const {
        if (jfif) return false;
        if (adobe >= 0) return adobe == 0;
        return cid[0] == 'R' && cid[1] == 'G' && cid[2] == 'B';
    }
};

// The end of an entropy-coded segment: the first marker that is neither a stuffed zero nor RSTn, less the fill bytes
// (0xFF, T.81 B.1.1.2) in front of it. An 0xFF of entropy data is always followed by a stuffed zero, so an 0xFF right
// before a marker is fill.
static size_t segment_end(const uint8_t *jpg, size_t len, size_t e) {
    const size_t e0 = e;
    const uint8_t *f = nullptr;
    while (e < len && (f = (const uint8_t *)memchr(jpg + e, 0xFF, len - e)) != nullptr) {
        e = (size_t)(f - jpg);
        if (e + 1 >= len) { e = len; break; }
        const uint8_t nx = jpg[e + 1];
        if (nx == 0x00 || (nx >= 0xD0 && nx <= 0xD7)) { e += 2; continue; }
        if (nx == 0xFF) { e += 1; continue; }
        break;
    }
    if (e > len || f == nullptr) e = len;
    while (e > e0 && jpg[e - 1] == 0xFF) e--;
    return e;
}

int parse_jpeg(const uint8_t *jpg, size_t len, JpegInfo *info) {
    static const uint8_t ZZ[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                                   41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                                   30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
    *info = JpegInfo();
    if (!jpg || len < 4 || jpg[0] != 0xFF || jpg[1] != 0xD8) return B2J_EFORMAT;
    uint16_t q[4][64];
    bool have_q[4] = {false, false, false, false};
    uint8_t hb[2][4][17], hv[2][4][256];
    bool have_h[2][4] = {{false, false, false, false}, {false, false, false, false}};
    memset(hb, 0, sizeof(hb));
    memset(hv, 0, sizeof(hv));
    int cid[3] = {0, 0, 0}, chv[3] = {0, 0, 0}, ctq[3] = {0, 0, 0}, ncomp = 0, ri = 0;
    int coef_bits[3][10];   // jdphuff.c coef_bits for zig-zag 0..9: the Al of the last scan that sent it, -1: none yet
    memset(coef_bits, 0xFF, sizeof(coef_bits));
    ColourMarkers cm;
    size_t p = 2;
    while (p + 2 <= len) {
        if (jpg[p] != 0xFF) return B2J_EFORMAT;
        const int m = jpg[p + 1];
        if (m == 0xFF) { p++; continue; }
        p += 2;
        if (m == 0x01 || (m >= 0xD0 && m <= 0xD8)) continue;
        if (m == 0xD9 || p + 2 > len) break;
        const int L = be16(jpg + p);
        if (L < 2 || p + L > len) return B2J_EFORMAT;
        const uint8_t *s = jpg + p + 2;
        int n = L - 2;
        switch (m) {
        case 0xDB:
            while (n > 0) {
                const int pq = s[0] >> 4, tq = s[0] & 15;
                const int sz = pq ? 128 : 64;
                if (tq > 3 || n < 1 + sz) return B2J_EFORMAT;
                for (int k = 0; k < 64; k++) q[tq][ZZ[k]] = (uint16_t)(pq ? be16(s + 1 + 2 * k) : s[1 + k]);
                have_q[tq] = true;
                s += 1 + sz; n -= 1 + sz;
            }
            break;
        case 0xC0: case 0xC1: case 0xC2:
            // a sequential file takes the last SOF before its scan; a progressive file has one
            if (ncomp && (info->progressive || m == 0xC2)) return B2J_EFORMAT;
            if (n < 9 || s[0] != 8 || (s[5] != 3 && s[5] != 1) || n < 6 + 3 * s[5]) return B2J_EFORMAT;
            info->progressive = m == 0xC2;
            info->H = be16(s + 1); info->W = be16(s + 3); ncomp = s[5];
            for (int c = 0; c < ncomp; c++) {
                cid[c] = s[6 + 3 * c]; chv[c] = s[7 + 3 * c]; ctq[c] = s[8 + 3 * c];
                if (ctq[c] > 3) return B2J_EFORMAT;   // jdinput.c latch_quant_tables: JERR_NO_QUANT_TABLE
            }
            if (ncomp == 1) { cid[1] = cid[2] = -1; ctq[1] = ctq[2] = ctq[0]; }   // no scan can name them; qt[1] = qt[0]
            break;
        case 0xC3: case 0xC5: case 0xC6: case 0xC7: case 0xC9: case 0xCA: case 0xCB: case 0xCD: case 0xCE: case 0xCF:
            return B2J_EFORMAT;  // lossless / hierarchical / arithmetic (SURVEY.md 8f N4)
        case 0xC4:
            while (n > 0) {
                const int tc = s[0] >> 4, th = s[0] & 15;
                if (tc > 1 || th > 3 || n < 17) return B2J_EFORMAT;
                int ns = 0;
                hb[tc][th][0] = 0;
                for (int l = 1; l <= 16; l++) { hb[tc][th][l] = s[l]; ns += s[l]; }
                if (ns > 256 || n < 17 + ns) return B2J_EFORMAT;
                // jdhuff.c jpeg_make_d_derived_tbl: a length may not hold more codes than the prefix code space leaves
                for (int l = 1, code = 0; l <= 16; l++) {
                    code += s[l];
                    if (code > (1 << l)) return B2J_EFORMAT;
                    code <<= 1;
                }
                memset(hv[tc][th], 0, 256);
                memcpy(hv[tc][th], s + 17, ns);
                have_h[tc][th] = true;
                s += 17 + ns; n -= 17 + ns;
            }
            break;
        case 0xDD:
            if (n < 2) return B2J_EFORMAT;
            ri = be16(s);
            break;
        case 0xDA: {
            if (info->scans.empty()) {   // the frame is final at the first scan, and so is the colour space (jpeg_read_header)
                if (ncomp == 3) {
                    if (chv[1] != 0x11 || chv[2] != 0x11 || ctq[1] != ctq[2] || cm.rgb(cid)) return B2J_EFORMAT;
                    info->hs = chv[0] >> 4; info->vs = chv[0] & 15;
                    static const int HS[5] = {1, 2, 1, 2, 4}, VS[5] = {1, 1, 2, 2, 1};
                    info->css = -1;
                    for (int i = 0; i < 5; i++) if (HS[i] == info->hs && VS[i] == info->vs) info->css = i;
                    if (info->css < 0) return B2J_EFORMAT;
                } else if (ncomp == 1) {   // one component (gray): its scans are non-interleaved, one block per MCU
                    info->css = B2J_CSS_GRAY; info->hs = info->vs = 1;
                } else {
                    return B2J_EFORMAT;    // no frame yet
                }
                if (info->W <= 0 || info->H <= 0) return B2J_EFORMAT;
            }
            if (n < 6) return B2J_EFORMAT;
            JpegScan sc;
            memset(&sc, 0, sizeof(sc));
            sc.ncomp = s[0];
            if (sc.ncomp < 1 || sc.ncomp > 3 || n < 4 + 2 * sc.ncomp) return B2J_EFORMAT;
            if (!info->progressive && sc.ncomp != ncomp) return B2J_EFORMAT;
            int td[3], ta[3];
            for (int i = 0; i < sc.ncomp; i++) {
                // a progressive scan names its components by id, a sequential one every component in frame order
                sc.comp[i] = -1;
                for (int c = 0; c < 3; c++) if (cid[c] == s[1 + 2 * i] && (info->progressive || c == i)) sc.comp[i] = c;
                td[i] = s[2 + 2 * i] >> 4; ta[i] = s[2 + 2 * i] & 15;
                if (sc.comp[i] < 0 || td[i] > 3 || ta[i] > 3) return B2J_EFORMAT;
                // interleaved scans: distinct components in frame order (jdinput.c would accept more orders)
                if (i > 0 && sc.comp[i] <= sc.comp[i - 1]) return B2J_EFORMAT;
                memcpy(sc.bits[0][i], hb[0][td[i]], 17); memcpy(sc.vals[0][i], hv[0][td[i]], 256);
                memcpy(sc.bits[1][i], hb[1][ta[i]], 17); memcpy(sc.vals[1][i], hv[1][ta[i]], 256);
            }
            if (info->progressive) {
                sc.Ss = s[1 + 2 * sc.ncomp]; sc.Se = s[2 + 2 * sc.ncomp];
                sc.Ah = s[3 + 2 * sc.ncomp] >> 4; sc.Al = s[3 + 2 * sc.ncomp] & 15;
                // jdphuff.c start_pass_phuff_decoder: a refinement scan refines by exactly one bit
                if (sc.Ss > sc.Se || sc.Se > 63 || (sc.Ss == 0 && sc.Se != 0) || (sc.Ss > 0 && sc.ncomp != 1) || sc.Al > 13 ||
                    (sc.Ah != 0 && sc.Al != sc.Ah - 1))
                    return B2J_EFORMAT;
                for (int i = 0; i < sc.ncomp; i++)
                    for (int k = sc.Ss; k <= sc.Se && k < 10; k++) coef_bits[sc.comp[i]][k] = sc.Al;
            } else {
                sc.Se = 63;
                if (sc.ncomp == 3 && (td[1] != td[2] || ta[1] != ta[2])) return B2J_EFORMAT;   // one table pair for Cb and Cr
            }
            // the tables the scan decodes with: DC for a first DC scan, AC for a band of AC coefficients
            for (int i = 0; i < sc.ncomp; i++)
                if ((sc.Ss == 0 && sc.Ah == 0 && !have_h[0][td[i]]) || (sc.Se > 0 && !have_h[1][ta[i]])) return B2J_EFORMAT;
            if (!have_q[ctq[0]] || !have_q[ctq[1]]) return B2J_EFORMAT;
            sc.restart_interval = ri;
            sc.seg_off = p + L;
            size_t e = sc.seg_off;
            if (!info->progressive && len >= e + 2 && jpg[len - 2] == 0xFF && jpg[len - 1] == 0xD9) {
                // the sequential files this engine and libjpeg write (one scan, EOI as the last two bytes): no 0xFF search
                e = len - 2;
                while (e > sc.seg_off && jpg[e - 1] == 0xFF) e--;   // fill bytes before EOI
            } else {
                e = segment_end(jpg, len, e);
            }
            sc.seg_len = e - sc.seg_off;
            if (info->scans.size() == 4096) return B2J_EFORMAT;
            try {
                info->scans.push_back(sc);
            } catch (const std::bad_alloc &) {
                return B2J_ENOMEM;
            }
            memcpy(info->qt[0], q[ctq[0]], 128); memcpy(info->qt[1], q[ctq[1]], 128);
            if (!info->progressive) return B2J_OK;
            p = e;
            continue;
        }
        default: cm.note(m, s, n); break;  // APPn, COM, ...
        }
        p += L;
    }
    // EOI, or the end of the bytes: a progressive file may end right after its last scan (a sequential one has returned)
    if (info->scans.empty()) return B2J_EFORMAT;
    // jdcoefct.c smoothing_ok (libjpeg-turbo 2.1 and later): every component's DC has been sent, the quantisers of
    // zig-zag 0..9 are non-zero, and some coefficient among zig-zag 1..9 is unfinished (never sent, or sent with Al > 0).
    // Smoothing then changes a component only where that component is unfinished: on gray output, only Y counts.
    bool ok = true, unfinished[3] = {false, false, false};
    for (int c = 0; c < ncomp; c++) {
        ok = ok && coef_bits[c][0] >= 0;
        for (int k = 0; k < 10; k++) ok = ok && info->qt[c > 0][ZZ[k]] != 0;
        for (int k = 1; k < 10; k++) unfinished[c] = unfinished[c] || coef_bits[c][k] != 0;
    }
    info->smoothed[0] = ok && (unfinished[0] || unfinished[1] || unfinished[2]);
    info->smoothed[1] = ok && unfinished[0];
    return B2J_OK;
}

size_t dec_tables_size() { return sizeof(DecTables); }

// jdhuff.c jpeg_make_d_derived_tbl. The parser has already rejected over-full tables; the bounds are checked again here
// because the tables index shared memory on the device.
int huff_derive(const uint8_t bits[17], const uint8_t vals[256], int lut_bits, uint16_t *lut, int32_t *maxcode, int32_t *valoff,
                uint8_t *vals_out) {
    memset(lut, 0, sizeof(uint16_t) << lut_bits);
    maxcode[0] = valoff[0] = 0;
    int code = 0, p = 0;
    for (int l = 1; l <= 16; l++) {
        const int n = bits[l];
        if (code + n > (1 << l) || p + n > 256) return B2J_EFORMAT;
        valoff[l] = p - code;
        for (int i = 0; i < n; i++, p++, code++) {
            if (l <= lut_bits) {
                const int lo = code << (lut_bits - l), cnt = 1 << (lut_bits - l);
                if (lo + cnt > (1 << lut_bits)) return B2J_EFORMAT;
                for (int j = 0; j < cnt; j++) lut[lo + j] = (uint16_t)((l << 8) | vals[p]);
            }
        }
        maxcode[l] = n ? code - 1 : -1;
        code <<= 1;
    }
    maxcode[17] = 0x7fffffff;
    memcpy(vals_out, vals, 256);
    return B2J_OK;
}

// the sequential decode tables: DC0, AC0 of Y and DC1, AC1 of Cb (Cr shares them; gray: Y's tables twice)
int dec_build_tables(const JpegInfo &info, void *dst) {
    DecTables *t = (DecTables *)dst;
    const JpegScan &sc = info.scans[0];
    for (int ti = 0; ti < 4; ti++) {
        const int k = ti & 1, c = ti >= 2 && sc.ncomp > 1 ? 1 : 0;
        if (huff_derive(sc.bits[k][c], sc.vals[k][c], DEC_LUT_BITS, t->lut[ti], t->maxcode[ti], t->valoff[ti], t->vals[ti]))
            return B2J_EFORMAT;
    }
    memcpy(t->q, info.qt, sizeof(t->q));
    return B2J_OK;
}

}  // namespace b2j
