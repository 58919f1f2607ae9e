// dec.h -- decoder interface internal to libb2jpeg.so (host parser + device pipeline)
#pragma once
#include <stddef.h>
#include <stdint.h>

#include "../../include/b2jpeg.h"
#include "common.cuh"

namespace b2j {

struct JpegInfo {
    int W, H, css, hs, vs;         // css B2J_CSS_GRAY: one component (hs = vs = 1 whatever its SOF says)
    int restart_interval;
    size_t scan_offset, scan_len;  // entropy-coded segment (stuffed bytes, up to the terminating marker)
    uint16_t qt[2][64];            // natural order: luma, chroma (gray: both the component's table)
    uint8_t bits[4][17];           // DC0, AC0, DC1, AC1 as used by Y / (Cb,Cr) (gray: the component's tables twice)
    uint8_t vals[4][256];
};

// jdmarker.c subset: baseline SOF0, 3 components, chroma 1x1, luma in {1x1,2x1,1x2,2x2,4x1}, one interleaved scan; or
// one component (any sampling factor: its single scan is non-interleaved, one block per MCU) -> css B2J_CSS_GRAY.
int parse_jpeg(const uint8_t *jpg, size_t len, JpegInfo *info);

struct Decoder;
Decoder *dec_create(int nblocks_cap, char *err, size_t errlen);
void dec_destroy(Decoder *d);
// careful = false: no host synchronisation inside (dec_check may then answer DEC_RETRY: run again with careful = true)
// d_scan_src != NULL: the scan's stuffed bytes are already in device memory (info.scan_len of them): nothing is uploaded
// gray_out: d_bgr receives one byte per pixel, the Y samples (JCS_GRAYSCALE; chroma blocks are decoded, not transformed)
// scale 2 / 4 / 8: d_bgr receives the image at 1 / scale (dec_kernels.h dec_scale_setup), 1: full size
int dec_run(Decoder *d, const uint8_t *jpg, size_t len, const JpegInfo &info, const Geom &g, uint8_t *d_bgr, size_t step,
            bool gray_out, cudaStream_t s, b2j_timings *tm, uint64_t *launches, bool careful, const uint8_t *d_scan_src = nullptr,
            int scale = 1);
constexpr int DEC_RETRY = 1;
int dec_check(Decoder *d, char *err, size_t errlen);   // synchronises the decode's stream
// optional: how host bytes reach the device (the API layer stages pageable memory through pinned buffers); the
// function returns a B2J_* status and must leave the copy ordered on stream s
typedef int (*dec_upload_fn)(void *user, uint8_t *d_dst, const uint8_t *src, size_t n, cudaStream_t s);
void dec_set_uploader(Decoder *d, dec_upload_fn fn, void *user);
void dec_set_spec_launches(Decoder *d, int n);   // speculative synchronisation launches (default 3)
const void *dec_coef_ptr(Decoder *d, size_t *bytes);

}  // namespace b2j

namespace b2j {

// ---- progressive (SOF2) streams: what the reference as shipped writes (ImageCompressorImpl.cu:28) -------------------
struct ProgScan {
    int ncomp, comp[3];            // components of the scan (indices 0 Y, 1 Cb, 2 Cr)
    int Ss, Se, Ah, Al;            // spectral selection, successive approximation
    int restart_interval;          // MCUs (interleaved) or blocks (one component) per interval, 0 = none
    size_t seg_off, seg_len;       // entropy-coded segment in the file (stuffed bytes, RSTn markers inside)
    uint8_t bits[2][3][17];        // [0 DC | 1 AC][component of the scan]: the tables in force at this SOS
    uint8_t vals[2][3][256];
};
struct ProgInfo {
    int W, H, css, hs, vs;         // as JpegInfo (css B2J_CSS_GRAY: one component)
    uint16_t qt[2][64];            // natural order: luma, chroma
    int nscans;
    ProgScan *scans;               // nscans entries (malloc'ed by parse_progressive, freed by prog_free)
};
// jdmarker.c for SOF2 files with three components, chroma 1x1, or one component; B2J_EFORMAT for anything else
int parse_progressive(const uint8_t *jpg, size_t len, ProgInfo *info);
void prog_free(ProgInfo *info);
// every scan is absorbed into the coefficient array in file order, then the baseline back end runs
int dec_run_progressive(Decoder *d, const uint8_t *jpg, size_t len, const ProgInfo &info, const Geom &g, uint8_t *d_bgr,
                        size_t step, bool gray_out, cudaStream_t s, uint64_t *launches, int scale = 1);

}  // namespace b2j
