// dec.h -- decoder interface internal to libb2jpeg.so (host parser + device pipeline)
#pragma once
#include <stddef.h>
#include <stdint.h>

#include <vector>

#include "../../include/b2jpeg.h"
#include "common.cuh"

namespace b2j {

// one scan: a sequential file has one (every component, Ss = 0, Se = 63, Ah = Al = 0), a progressive file one per SOS
struct JpegScan {
    int ncomp, comp[3];            // components of the scan (indices 0 Y, 1 Cb, 2 Cr)
    int Ss, Se, Ah, Al;            // spectral selection, successive approximation
    int restart_interval;          // MCUs (interleaved) or blocks (one component) per interval, 0 = none
    size_t seg_off, seg_len;       // entropy-coded segment in the file (stuffed bytes, RSTn markers inside)
    uint8_t bits[2][3][17];        // [0 DC | 1 AC][component of the scan]: the tables in force at this SOS
    uint8_t vals[2][3][256];
};
struct JpegInfo {
    int W, H, css, hs, vs;         // css B2J_CSS_GRAY: one component (hs = vs = 1 whatever its SOF says)
    bool progressive;              // SOF2: scans up to EOI; else SOF0 / SOF1: the first scan only
    uint16_t qt[2][64];            // natural order: luma, chroma (gray: both the component's table), as at the last SOS
    std::vector<JpegScan> scans;
    // a progressive file that leaves low-frequency coefficients unfinished: libjpeg-turbo block-smooths such output
    // (jdcoefct.c smoothing_ok), which this decoder does not restate, so the decode entry points refuse it.
    // [0]: BGR output (any component unfinished), [1]: gray output (the Y plane: Y unfinished)
    bool smoothed[2];
};

// jdmarker.c subset: SOF0 / SOF1 / SOF2, 3 components, chroma 1x1, luma in {1x1,2x1,1x2,2x2,4x1}; or one component (any
// sampling factor, laid out one block per MCU) -> css B2J_CSS_GRAY. A sequential file has one interleaved scan (Cb and
// Cr share their tables) and is parsed up to it; a progressive file is parsed up to EOI (at most 4096 scans).
int parse_jpeg(const uint8_t *jpg, size_t len, JpegInfo *info);

struct Decoder;
Decoder *dec_create(int nblocks_cap, char *err, size_t errlen);
void dec_destroy(Decoder *d);
// sequential files (info.scans[0]):
// careful = false: no host synchronisation inside (dec_check may then answer DEC_RETRY: run again with careful = true)
// d_scan_src != NULL: the scan's stuffed bytes are already in device memory (seg_len of them): nothing is uploaded
// gray_out: d_bgr receives one byte per pixel, the Y samples (JCS_GRAYSCALE; chroma blocks are decoded, not transformed)
// scale 2 / 4 / 8: d_bgr receives the image at 1 / scale (dec_kernels.h dec_scale_setup), 1: full size
// region != NULL: {x, y, w, h} of the output (w = 0: all of it), inside the output size; d_bgr receives that rectangle
// (its pixel (x, y) at d_bgr) and nothing else (dec_kernels.h DecWin)
int dec_run(Decoder *d, const uint8_t *jpg, size_t len, const JpegInfo &info, const Geom &g, uint8_t *d_bgr, size_t step,
            bool gray_out, cudaStream_t s, b2j_timings *tm, uint64_t *launches, bool careful, const uint8_t *d_scan_src = nullptr,
            int scale = 1, const int *region = nullptr);
constexpr int DEC_RETRY = 1;
int dec_check(Decoder *d, char *err, size_t errlen);   // synchronises the decode's stream
// optional: how host bytes reach the device (the API layer stages pageable memory through pinned buffers); the
// function returns a B2J_* status and must leave the copy ordered on stream s
typedef int (*dec_upload_fn)(void *user, uint8_t *d_dst, const uint8_t *src, size_t n, cudaStream_t s);
void dec_set_uploader(Decoder *d, dec_upload_fn fn, void *user);
void dec_set_spec_launches(Decoder *d, int n);   // speculative synchronisation launches (default 3)
const void *dec_coef_ptr(Decoder *d, size_t *bytes);

// progressive files (SOF2, what the reference as shipped writes, ImageCompressorImpl.cu:28): every scan is absorbed into
// the coefficient array in file order, then the back end of dec_run runs
int dec_run_progressive(Decoder *d, const uint8_t *jpg, size_t len, const JpegInfo &info, const Geom &g, uint8_t *d_bgr,
                        size_t step, bool gray_out, cudaStream_t s, uint64_t *launches, int scale = 1, const int *region = nullptr);

}  // namespace b2j
