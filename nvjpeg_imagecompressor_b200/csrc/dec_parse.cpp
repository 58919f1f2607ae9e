// dec_parse.cpp -- host-side marker parser (the reference does this with nvjpegGetImageInfo + nvjpegJpegStreamParse,
// ImageCompressorImpl.cu:335,362; semantics follow libjpeg jdmarker.c for the baseline subset listed in dec.h).
#include <stdlib.h>
#include <string.h>

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
    memset(info, 0, sizeof(*info));
    if (!jpg || len < 4 || jpg[0] != 0xFF || jpg[1] != 0xD8) return B2J_EFORMAT;
    uint16_t q[4][64];
    bool have_q[4] = {false, false, false, false};
    uint8_t hb[2][4][17], hv[2][4][256];
    bool have_h[2][4] = {{false, false, false, false}, {false, false, false, false}};
    memset(hb, 0, sizeof(hb));
    memset(hv, 0, sizeof(hv));
    int cid[3] = {0, 0, 0}, chv[3] = {0, 0, 0}, ctq[3] = {0, 0, 0}, ncomp = 0;
    ColourMarkers cm;
    size_t p = 2;
    while (p + 4 <= len) {
        if (jpg[p] != 0xFF) return B2J_EFORMAT;
        const int m = jpg[p + 1];
        if (m == 0xFF) { p++; continue; }
        p += 2;
        if (m == 0x01 || (m >= 0xD0 && m <= 0xD8)) continue;
        if (m == 0xD9) return B2J_EFORMAT;
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
        case 0xC0: case 0xC1:
            if (n < 9 || s[0] != 8 || (s[5] != 3 && s[5] != 1) || n < 6 + 3 * s[5]) return B2J_EFORMAT;
            info->H = be16(s + 1); info->W = be16(s + 3); ncomp = s[5];
            for (int c = 0; c < ncomp; c++) {
                cid[c] = s[6 + 3 * c]; chv[c] = s[7 + 3 * c]; ctq[c] = s[8 + 3 * c];
                if (ctq[c] > 3) return B2J_EFORMAT;   // jdinput.c latch_quant_tables: JERR_NO_QUANT_TABLE
            }
            break;
        case 0xC2: case 0xC3: case 0xC5: case 0xC6: case 0xC7: case 0xC9: case 0xCA: case 0xCB: case 0xCD: case 0xCE: case 0xCF:
            return B2J_EFORMAT;  // progressive / lossless / arithmetic (SURVEY.md 8f N4)
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
            info->restart_interval = be16(s);
            break;
        case 0xDA: {
            if (ncomp == 1) {   // one component (gray): one non-interleaved scan, laid out 1x1 whatever the SOF says
                if (n < 6 || s[0] != 1 || s[1] != cid[0]) return B2J_EFORMAT;
                const int td = s[2] >> 4, ta = s[2] & 15;
                if (td > 3 || ta > 3 || !have_h[0][td] || !have_h[1][ta] || !have_q[ctq[0]]) return B2J_EFORMAT;
                if (info->W <= 0 || info->H <= 0) return B2J_EFORMAT;
                info->css = B2J_CSS_GRAY; info->hs = info->vs = 1;
                for (int t = 0; t < 2; t++) memcpy(info->qt[t], q[ctq[0]], 128);
                for (int t = 0; t < 4; t += 2) {
                    memcpy(info->bits[t], hb[0][td], 17); memcpy(info->vals[t], hv[0][td], 256);
                    memcpy(info->bits[t + 1], hb[1][ta], 17); memcpy(info->vals[t + 1], hv[1][ta], 256);
                }
            }
            if (ncomp != 3 && ncomp != 1) return B2J_EFORMAT;
            if (ncomp == 3 && (n < 10 || s[0] != 3)) return B2J_EFORMAT;
            int td[3], ta[3];
            for (int c = 0; c < 3 && ncomp == 3; c++) {
                if (s[1 + 2 * c] != cid[c]) return B2J_EFORMAT;
                td[c] = s[2 + 2 * c] >> 4; ta[c] = s[2 + 2 * c] & 15;
                if (td[c] > 3 || ta[c] > 3 || !have_h[0][td[c]] || !have_h[1][ta[c]]) return B2J_EFORMAT;
            }
            if (ncomp == 3) {
                if (cm.rgb(cid)) return B2J_EFORMAT;
                if (chv[1] != 0x11 || chv[2] != 0x11 || td[1] != td[2] || ta[1] != ta[2] || ctq[1] != ctq[2]) return B2J_EFORMAT;
                if (!have_q[ctq[0]] || !have_q[ctq[1]]) return B2J_EFORMAT;
                info->hs = chv[0] >> 4; info->vs = chv[0] & 15;
                static const int HS[5] = {1, 2, 1, 2, 4}, VS[5] = {1, 1, 2, 2, 1};
                info->css = -1;
                for (int i = 0; i < 5; i++) if (HS[i] == info->hs && VS[i] == info->vs) info->css = i;
                if (info->css < 0 || info->W <= 0 || info->H <= 0) return B2J_EFORMAT;
                memcpy(info->qt[0], q[ctq[0]], 128); memcpy(info->qt[1], q[ctq[1]], 128);
                memcpy(info->bits[0], hb[0][td[0]], 17); memcpy(info->vals[0], hv[0][td[0]], 256);
                memcpy(info->bits[1], hb[1][ta[0]], 17); memcpy(info->vals[1], hv[1][ta[0]], 256);
                memcpy(info->bits[2], hb[0][td[1]], 17); memcpy(info->vals[2], hv[0][td[1]], 256);
                memcpy(info->bits[3], hb[1][ta[1]], 17); memcpy(info->vals[3], hv[1][ta[1]], 256);
            }
            info->scan_offset = p + L;
            // the entropy-coded segment (segment_end). Fast path for the files this engine and libjpeg write (one scan,
            // EOI as the last two bytes): no 0xFF search at all.
            size_t e = info->scan_offset;
            if (len >= e + 2 && jpg[len - 2] == 0xFF && jpg[len - 1] == 0xD9) {
                e = len - 2;
                while (e > info->scan_offset && jpg[e - 1] == 0xFF) e--;   // fill bytes before EOI
            } else {
                e = segment_end(jpg, len, e);
            }
            info->scan_len = e - info->scan_offset;
            return B2J_OK;
        }
        default: cm.note(m, s, n); break;  // APPn, COM, ...
        }
        p += L;
    }
    return B2J_EFORMAT;
}

// ---------------------------------------------------------------------------------------------------------------
// Progressive files (SOF2): frame header, tables as they stand at every SOS, one ProgScan per scan.
void prog_free(ProgInfo *info) { if (info && info->scans) { free(info->scans); info->scans = nullptr; info->nscans = 0; } }

int parse_progressive(const uint8_t *jpg, size_t len, ProgInfo *info) {
    static const uint8_t ZZ[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                                   41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                                   30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
    memset(info, 0, sizeof(*info));
    if (!jpg || len < 4 || jpg[0] != 0xFF || jpg[1] != 0xD8) return B2J_EFORMAT;
    uint16_t q[4][64];
    bool have_q[4] = {false, false, false, false};
    static thread_local uint8_t hb[2][4][17], hv[2][4][256];
    bool have_h[2][4] = {{false, false, false, false}, {false, false, false, false}};
    memset(hb, 0, sizeof(hb));
    memset(hv, 0, sizeof(hv));
    int cid[3] = {0, 0, 0}, chv[3] = {0, 0, 0}, ctq[3] = {0, 0, 0};
    int ri = 0, cap = 0;
    bool have_sof = false;
    ColourMarkers cm;
    size_t p = 2;
    int rc = B2J_EFORMAT;
    while (p + 2 <= len) {
        if (jpg[p] != 0xFF) break;
        const int m = jpg[p + 1];
        if (m == 0xFF) { p++; continue; }
        p += 2;
        if (m == 0x01 || (m >= 0xD0 && m <= 0xD8)) continue;
        if (m == 0xD9) { rc = (have_sof && info->nscans > 0) ? B2J_OK : B2J_EFORMAT; break; }
        if (p + 2 > len) break;
        const int L = be16(jpg + p);
        if (L < 2 || p + L > len) break;
        const uint8_t *s = jpg + p + 2;
        int n = L - 2;
        bool bad = false;
        if (m == 0xDB) {
            while (n > 0) {
                const int pq = s[0] >> 4, tq = s[0] & 15;
                const int sz = pq ? 128 : 64;
                if (tq > 3 || n < 1 + sz) { bad = true; break; }
                for (int k = 0; k < 64; k++) q[tq][ZZ[k]] = (uint16_t)(pq ? be16(s + 1 + 2 * k) : s[1 + k]);
                have_q[tq] = true;
                s += 1 + sz; n -= 1 + sz;
            }
        } else if (m == 0xC2) {
            if (have_sof || n < 9 || s[0] != 8 || (s[5] != 3 && s[5] != 1) || n < 6 + 3 * s[5]) { bad = true; }
            else if (s[5] == 1) {   // one component (gray): any sampling factor, laid out 1x1
                info->H = be16(s + 1); info->W = be16(s + 3);
                cid[0] = s[6]; ctq[0] = ctq[1] = ctq[2] = s[8];
                cid[1] = cid[2] = -1;   // no scan can name them
                info->hs = info->vs = 1; info->css = B2J_CSS_GRAY;
                if (info->W <= 0 || info->H <= 0 || ctq[0] > 3) bad = true;
                have_sof = !bad;
            } else {
                info->H = be16(s + 1); info->W = be16(s + 3);
                for (int c = 0; c < 3; c++) { cid[c] = s[6 + 3 * c]; chv[c] = s[7 + 3 * c]; ctq[c] = s[8 + 3 * c]; }
                if (chv[1] != 0x11 || chv[2] != 0x11 || ctq[1] != ctq[2] || ctq[0] > 3 || ctq[1] > 3) bad = true;
                info->hs = chv[0] >> 4; info->vs = chv[0] & 15;
                static const int HS[5] = {1, 2, 1, 2, 4}, VS[5] = {1, 1, 2, 2, 1};
                info->css = -1;
                for (int i = 0; i < 5; i++) if (HS[i] == info->hs && VS[i] == info->vs) info->css = i;
                if (info->css < 0 || info->W <= 0 || info->H <= 0) bad = true;
                have_sof = !bad;
            }
        } else if ((m >= 0xC0 && m <= 0xCF) && m != 0xC4 && m != 0xC8 && m != 0xCC) {
            bad = true;   // not a progressive Huffman frame
        } else if (m == 0xC4) {
            while (n > 0) {
                const int tc = s[0] >> 4, th = s[0] & 15;
                if (tc > 1 || th > 3 || n < 17) { bad = true; break; }
                int ns = 0, code = 0;
                for (int l = 1; l <= 16; l++) {
                    hb[tc][th][l] = s[l]; ns += s[l];
                    code += s[l];
                    if (code > (1 << l)) bad = true;   // more codes than the prefix space leaves
                    code <<= 1;
                }
                if (bad || ns > 256 || n < 17 + ns) { bad = true; break; }
                memset(hv[tc][th], 0, 256);
                memcpy(hv[tc][th], s + 17, ns);
                have_h[tc][th] = true;
                s += 17 + ns; n -= 17 + ns;
            }
        } else if (m == 0xDD) {
            if (n < 2) bad = true; else ri = be16(s);
        } else if (m == 0xDA) {
            // the colour space is settled by the markers before the first scan (jpeg_read_header)
            if (!have_sof || n < 6 || (info->nscans == 0 && info->css != B2J_CSS_GRAY && cm.rgb(cid))) { bad = true; }
            else {
                ProgScan sc;
                memset(&sc, 0, sizeof(sc));
                sc.ncomp = s[0];
                if (sc.ncomp < 1 || sc.ncomp > 3 || n < 4 + 2 * sc.ncomp) bad = true;
                for (int i = 0; !bad && i < sc.ncomp; i++) {
                    sc.comp[i] = -1;
                    for (int c = 0; c < 3; c++) if (cid[c] == s[1 + 2 * i]) sc.comp[i] = c;
                    const int td = s[2 + 2 * i] >> 4, ta = s[2 + 2 * i] & 15;
                    if (sc.comp[i] < 0 || td > 3 || ta > 3) { bad = true; break; }
                    memcpy(sc.bits[0][i], hb[0][td], 17); memcpy(sc.vals[0][i], hv[0][td], 256);
                    memcpy(sc.bits[1][i], hb[1][ta], 17); memcpy(sc.vals[1][i], hv[1][ta], 256);
                    sc.comp[i] |= (have_h[0][td] ? 0 : 0x100) | (have_h[1][ta] ? 0 : 0x200);   // checked below against Ss
                }
                if (!bad) {
                    sc.Ss = s[1 + 2 * sc.ncomp]; sc.Se = s[2 + 2 * sc.ncomp];
                    sc.Ah = s[3 + 2 * sc.ncomp] >> 4; sc.Al = s[3 + 2 * sc.ncomp] & 15;
                    if (sc.Ss > sc.Se || sc.Se > 63 || (sc.Ss == 0 && sc.Se != 0) || (sc.Ss > 0 && sc.ncomp != 1) || sc.Al > 13 || sc.Ah > 13) bad = true;
                    for (int i = 0; !bad && i < sc.ncomp; i++) {
                        const bool need_dc = sc.Ss == 0 && sc.Ah == 0, need_ac = sc.Ss > 0;
                        if ((need_dc && (sc.comp[i] & 0x100)) || (need_ac && (sc.comp[i] & 0x200))) bad = true;
                        sc.comp[i] &= 0xFF;
                    }
                    // three distinct components in frame order for interleaved scans (jdinput.c would accept more orders)
                    for (int i = 1; !bad && i < sc.ncomp; i++) if (sc.comp[i] <= sc.comp[i - 1]) bad = true;
                    if (!have_q[ctq[0]] || !have_q[ctq[1]]) bad = true;
                }
                if (!bad) {
                    sc.restart_interval = ri;
                    sc.seg_off = p + L;
                    const size_t e = segment_end(jpg, len, sc.seg_off);
                    sc.seg_len = e - sc.seg_off;
                    if (info->nscans == cap) {
                        cap = cap ? cap * 2 : 16;
                        if (cap > 4096) { bad = true; }
                        else {
                            ProgScan *ns2 = (ProgScan *)realloc(info->scans, sizeof(ProgScan) * cap);
                            if (!ns2) { prog_free(info); return B2J_ENOMEM; }
                            info->scans = ns2;
                        }
                    }
                    if (!bad) {
                        info->scans[info->nscans++] = sc;
                        memcpy(info->qt[0], q[ctq[0]], 128); memcpy(info->qt[1], q[ctq[1]], 128);
                        p = e;
                        continue;
                    }
                }
            }
        } else {
            cm.note(m, s, n);   // APPn, COM, ...
        }
        if (bad) break;
        p += L;
    }
    if (rc != B2J_OK && have_sof && info->nscans > 0 && p + 2 > len) rc = B2J_OK;   // no EOI after the last scan: tolerated
    if (rc != B2J_OK) prog_free(info);
    return rc;
}

size_t dec_tables_size() { return sizeof(DecTables); }

// host-side construction of the decode tables (jdhuff.c jpeg_make_d_derived_tbl). parse_jpeg has already rejected
// over-full tables; the bounds are checked again here because the tables index shared memory on the device.
int dec_build_tables(const JpegInfo &info, void *dst) {
    DecTables *t = (DecTables *)dst;
    memset(t, 0, sizeof(*t));
    for (int ti = 0; ti < 4; ti++) {
        int code = 0, p = 0;
        for (int l = 1; l <= 16; l++) {
            const int n = info.bits[ti][l];
            if (code + n > (1 << l) || p + n > 256) return B2J_EFORMAT;
            t->valoff[ti][l] = p - code;
            for (int i = 0; i < n; i++, p++, code++) {
                if (l <= DEC_LUT_BITS) {
                    const int lo = code << (DEC_LUT_BITS - l), cnt = 1 << (DEC_LUT_BITS - l);
                    if (lo + cnt > (1 << DEC_LUT_BITS)) return B2J_EFORMAT;
                    for (int j = 0; j < cnt; j++) t->lut[ti][lo + j] = (uint16_t)((l << 8) | info.vals[ti][p]);
                }
            }
            t->maxcode[ti][l] = n ? code - 1 : -1;
            code <<= 1;
        }
        t->maxcode[ti][17] = 0x7fffffff;
        memcpy(t->vals[ti], info.vals[ti], 256);
    }
    memcpy(t->q, info.qt, sizeof(t->q));
    return B2J_OK;
}

}  // namespace b2j
