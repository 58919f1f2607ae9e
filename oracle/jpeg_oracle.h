/*
 * jpeg_oracle.h -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * CPU restatement (plain C) of the baseline-JPEG arithmetic that the reference's hot path
 * delegates to a codec library (reference call sites: src/ImageCompressorDll/ImageCompressorImpl.cu:280
 * nvjpegEncodeImage, :364-366 nvjpegDecodeJpeg*). The north-star pins bit-exactness to libjpeg-turbo
 * (DCT_ISLOW, no restart markers), so this file restates libjpeg-turbo 3.1.2's published algorithm
 * (jccolor.c, jcsample.c, jcprepct.c, jfdctint.c, jcdctmgr.c, jccoefct.c, jchuff.c, jcparam.c,
 * jcmarker.c / jdhuff.c, jidctint.c, jdsample.c, jdcolor.c) as written down in SURVEY.md Appendix A.
 *
 * Parity pin: tests/test_oracle_golden.py, test_oracle_gray.py, test_oracle_scaled.py and test_prog_streams.py compare
 * the functions here byte-for-byte with cv2.imencode / cv2.imdecode (OpenCV 4.13.0 wheel = libjpeg-turbo 3.1.2), and
 * tests/golden/ holds committed digests produced by that library (tests/golden/make_golden*.py).
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / reference leg may link or call this.
 */
#ifndef JPEG_ORACLE_H_
#define JPEG_ORACLE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* chroma subsampling codes shared with include/b2jpeg.h; GRAY: one component (orc_geometry refuses it) */
enum { ORC_CSS_444 = 0, ORC_CSS_422 = 1, ORC_CSS_440 = 2, ORC_CSS_420 = 3, ORC_CSS_411 = 4, ORC_CSS_GRAY = 6 };

typedef struct {
    int W, H, css;
    int hs, vs;          /* luma sampling factors (chroma is 1x1) */
    int mcux, mcuy;      /* MCU grid */
    int bpm;             /* blocks per MCU = hs*vs + 2 (gray: 1) */
    int wib[3], hib[3];  /* per-component width/height in blocks (real data) */
    int dw[3], dh[3];    /* per-component true downsampled size in samples */
    long long nblocks;   /* mcux*mcuy*bpm (scan order) */
} orc_geom;

int  orc_geometry(int W, int H, int css, orc_geom *g);

/* quant tables in NATURAL order: qt[0] luma, qt[1] chroma  (jcparam.c jpeg_set_quality) */
void orc_quant_tables(int quality, uint16_t qt[2][64]);

/* synthetic generator of SURVEY.md Appendix B; out is H*W*3 BGR, tightly packed */
void orc_synth(int W, int H, uint32_t seed, int amp, uint8_t *out);
/* same generator, rows [y0, y0+rows) only */
void orc_synth_rows(int W, int H, int y0, int rows, uint32_t seed, int amp, uint8_t *out);

/* Stage 1+2: BGR -> quantised coefficients, scan order (MCU raster; Y blocks row-major, Cb, Cr),
 * 64 int16 per block in ZIG-ZAG order. coef must hold g.nblocks*64 int16. */
int  orc_forward(const uint8_t *bgr, size_t step, int W, int H, int css, int quality, int16_t *coef);

/* Stage 3: symbol histograms. hist[4][257]: DC0, AC0, DC1, AC1 (index 256 unused, left 0). bpm 1: one component,
 * counted as the last component (DC1, AC1); orc_entropy_bits codes it with tables 2 / 3 likewise.
 * pred_in/pred_out: optional DC predictors per component at strip start/end (NULL = 0 / ignored). */
void orc_histogram(const int16_t *coef, long long nblocks, int bpm, const int16_t *pred_in,
                   uint32_t hist[4][257]);

/* jpeg_gen_optimal_table: freq[257] (freq[256] is set to 1 inside) -> bits[1..16] in bits[17], huffval[256];
 * returns number of symbols. */
int  orc_gen_optimal_table(const uint32_t freq_in[257], uint8_t bits[17], uint8_t huffval[256]);

/* standard Annex-K tables: idx 0 DC0, 1 AC0, 2 DC1, 3 AC1 */
int  orc_std_table(int idx, uint8_t bits[17], uint8_t huffval[256]);

/* derive code/size per symbol from bits/huffval (Annex C) */
void orc_derive_codes(const uint8_t bits[17], const uint8_t huffval[256], uint16_t code[256], uint8_t size[256]);

/* Stage 4: entropy-code scan-order coefficients. Produces the UNSTUFFED bit string (MSB first) into
 * out (capacity cap bytes, zero-filled by the callee) and its length in bits. No padding applied. */
int  orc_entropy_bits(const int16_t *coef, long long nblocks, int bpm, const int16_t *pred_in,
                      const uint8_t bits[4][17], const uint8_t vals[4][256],
                      uint8_t *out, size_t cap, uint64_t *nbits);

/* Stuff a bit string: pad the last partial byte with 1-bits, insert 0x00 after every 0xFF. */
size_t orc_stuff(const uint8_t *in, uint64_t nbits, uint8_t *out, size_t cap);

/* JFIF headers exactly as jcmarker.c writes them (SOI .. SOS). returns length. */
size_t orc_headers(int W, int H, int css, const uint16_t qt[2][64], const uint8_t bits[4][17],
                   const uint8_t vals[4][256], uint8_t *out, size_t cap);

/* Whole encoder: returns 0 on success */
int  orc_encode(const uint8_t *bgr, size_t step, int W, int H, int css, int quality, int optimize,
                uint8_t *out, size_t cap, size_t *len);
/* Same with restart markers every `restart_interval` MCUs (0 = none): DRI before SOS, RSTn between the intervals,
 * DC predictors and the bit buffer restart (jchuff.c emit_restart). Pinned against cv2 IMWRITE_JPEG_RST_INTERVAL.
 * css ORC_CSS_GRAY: one component (JCS_GRAYSCALE) from 8-bit samples with row pitch `step`; DQT 0, SOF0 and SOS with
 * one component, DHT DC0 and AC0; the restart interval counts blocks (one block per MCU). */
int  orc_encode_rst(const uint8_t *px, size_t step, int W, int H, int css, int quality, int optimize,
                    int restart_interval, uint8_t *out, size_t cap, size_t *len);

/* Parsed header info */
typedef struct {
    int W, H, css;        /* css = -1 if the sampling is not one of the five supported */
    int hs, vs;
    int restart_interval;
    size_t scan_offset;   /* first byte of entropy-coded data */
    size_t scan_len;      /* bytes of entropy-coded data (up to, excluding, EOI marker) */
    uint16_t qt[2][64];   /* natural order, as used by comp 0 / comps 1,2 */
    uint8_t bits[4][17];  /* DC0, AC0, DC1, AC1 as used by Y / chroma */
    uint8_t vals[4][256];
} orc_info;

/* Headers of a three-component sequential file up to its (only) scan; -8 for a progressive file, -7 for one with one
 * component. */
int  orc_parse(const uint8_t *jpg, size_t len, orc_info *info);

/* Decode entropy data to scan-order quantised coefficients (zig-zag order), DC already un-differenced. */
int  orc_decode_coefs(const uint8_t *jpg, size_t len, const orc_info *info, int16_t *coef);

/* Stage 5: coefficients of orc_decode_coefs -> BGR (islow IDCT, fancy upsampling, jdcolor) */
int  orc_inverse(const int16_t *coef, const orc_info *info, uint8_t *bgr, size_t step);

/* Progressive (SOF2) encode: jpeg_simple_progression's 10 scans, optimal tables per scan (jcphuff.c); what
 * cv2.imencode(IMWRITE_JPEG_PROGRESSIVE) writes and the mode the reference hard-codes (ImageCompressorImpl.cu:28). */
int  orc_encode_progressive(const uint8_t *bgr, size_t step, int W, int H, int css, int quality, uint8_t *out,
                            size_t cap, size_t *len);

/* The decoders read sequential (SOF0/1) and progressive (SOF2) files with one or three components; a progressive
 * file's scans are all absorbed (jdphuff.c) before the one back end runs. *W, *H: the output size; the output may be
 * NULL to query it. 0 on success; -18 for a progressive file libjpeg would block-smooth (an output component's
 * low-frequency coefficients unfinished); other negative values: a file the product refuses. */

/* what libjpeg returns with scale_num = 1, scale_denom = d (1, 2, 4, 8; else -20; cv2 IMREAD_REDUCED_*_d): BGR
 * (H', W', 3) or, with gray_out, the luma plane (H', W') (JCS_GRAYSCALE: no chroma IDCT, upsampling or colour
 * conversion), row pitch `step`. Colour output of a one-component file: -21. */
int  orc_decode_output(const uint8_t *jpg, size_t len, int denom, int gray_out, uint8_t *out, size_t step, int *W, int *H);
/* full-size BGR (IMREAD_COLOR): orc_decode_output(jpg, len, 1, 0, ...) */
int  orc_decode(const uint8_t *jpg, size_t len, uint8_t *bgr, size_t step, int *W, int *H);
/* orc_decode of progressive files only (-8 otherwise) */
int  orc_decode_progressive(const uint8_t *jpg, size_t len, uint8_t *bgr, size_t step, int *W, int *H);

/* a-12 definitions (SURVEY.md 8a-12): mode 0 = absdiff, 1 = clamp(a-b+128) */
void   orc_diff(const uint8_t *a, const uint8_t *b, size_t n, int mode, uint8_t *out);
uint64_t orc_ssd(const uint8_t *a, const uint8_t *b, size_t n);
double orc_psnr(const uint8_t *a, const uint8_t *b, size_t n);

#ifdef __cplusplus
}
#endif
#endif
