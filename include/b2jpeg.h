/*
 * b2jpeg.h -- C-ABI of the B200-native JPEG engine (libb2jpeg.so).
 *
 * This is the drop-in boundary for the reference's hot path. Every entry point names the reference
 * interface it replaces (paths relative to the reference repository, OroChippw/Nvjpeg-ImageCompressor):
 *
 *   b2j_create / b2j_destroy      NvjpegCompressRunnerImpl::initCompressEnv / initDecodeEnv /
 *                                 destoryCompressEnv / destoryDecodeEnv
 *                                 (src/ImageCompressorDll/ImageCompressorImpl.cu:19-45, 47-65, 67-95, 97-117)
 *   b2j_encode                    NvjpegCompressRunnerImpl::CompressWorker  (ImageCompressorImpl.cu:269-294:
 *                                 cv::split + 3x cudaMemcpy + nvjpegEncodeImage + nvjpegEncodeRetrieveBitstream)
 *   b2j_encode_device             the cudaEvent bracket of the same function (ImageCompressorImpl.cu:279-281):
 *                                 input already on the device, bitstream left on the device
 *   b2j_decode / b2j_peek         NvjpegCompressRunnerImpl::DecodeWorker (ImageCompressorImpl.cu:311-385:
 *                                 nvjpegGetImageInfo, nvjpegDecodeJpegHost/TransferToDevice/Device) and
 *                                 getCVImageOnCPU (:184-232; the planar->interleaved step is fused into the store)
 *   b2j_diff / b2j_psnr /         the README's "difference map / secondary compression / PSNR" bullet
 *   b2j_secondary                 (README.md:8, PSNR column README.md:45) -- absent from the reference code,
 *                                 defined in SURVEY.md section 8 row a-12
 *
 * Conventions: plain pointers and sizes only (no cv::Mat, no torch types); pixels are 8-bit BGR interleaved
 * (cv::Mat CV_8UC3) with a row pitch `step >= 3 * width` in bytes -- on a context created with css = B2J_CSS_GRAY they
 * are 8-bit single-channel rows (cv::Mat CV_8UC1) with `step >= width`, wherever this header says "bgr"; every function returns 0 on success or a negative
 * B2J_E* code and never calls exit() (the reference's CHECK_CUDA/CHECK_NVJPEG exit(1),
 * ImageCompressorImpl.cuh:16-34, is deliberately not reproduced). One context = one encoder/decoder state on
 * one GPU, not thread-safe, synchronous at return unless stated otherwise (as the reference,
 * SURVEY.md 8b "Threading").
 */
#ifndef B2JPEG_H_
#define B2JPEG_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define B2J_API __declspec(dllexport)
#else
#define B2J_API __attribute__((visibility("default")))
#endif

/* nvjpegChromaSubsampling_t values the reference's README sweeps (README.md:44-51), and NVJPEG_CSS_GRAY (5 is not valid).
 * A B2J_CSS_GRAY context works on one byte per pixel:
 *   encode: the one-component stream libjpeg-turbo writes for a grayscale image (one DQT, SOF0 with one component,
 *           DC0/AC0 only; restart intervals of b2j_set_restart_rows rows of blocks);
 *   decode: a one-component file (baseline, restart markers, progressive; any sampling factor in its SOF) as libjpeg
 *           decodes it, and the Y plane of a three-component file (libjpeg's JCS_GRAYSCALE output);
 *   the strip / peer / multi-GPU encoders, b2j_reconstruct_* and b2j_secondary* refuse it with B2J_EINVAL.
 * Every other context refuses one-component files with B2J_EFORMAT; b2j_peek reports them as B2J_CSS_GRAY. */
enum { B2J_CSS_444 = 0, B2J_CSS_422 = 1, B2J_CSS_440 = 2, B2J_CSS_420 = 3, B2J_CSS_411 = 4, B2J_CSS_GRAY = 6 };

enum {
    B2J_OK = 0,
    B2J_EINVAL = -1,     /* bad argument */
    B2J_ECUDA = -2,      /* CUDA runtime error (b2j_last_error has the text) */
    B2J_ENOMEM = -3,
    B2J_ECAPACITY = -4,  /* output buffer too small */
    B2J_EFORMAT = -5,    /* not a JPEG this decoder handles (or a one-component file on a colour context) */
    B2J_EINTERNAL = -6,  /* a device-side consistency check failed */
    B2J_ESIZE = -7       /* image does not match the context's width/height */
};

/* b2j_diff modes */
enum { B2J_DIFF_ABS = 0, B2J_DIFF_OFFSET128 = 1 };

typedef struct b2j_ctx b2j_ctx;

/* Mirrors NvjpegCompressRunner's constructor (ImageCompressor.h:27) plus the sampling factor the reference
 * hard-codes at ImageCompressorImpl.cu:31. */
typedef struct b2j_params {
    int width;     /* default 8320  */
    int height;    /* default 40000 */
    int quality;   /* default 95    */
    int optimize;  /* optimized Huffman, default 1 */
    int css;       /* B2J_CSS_*, README default 422 */
    int device;    /* CUDA device ordinal; -1 = current device */
    int flags;     /* B2J_FLAG_* */
} b2j_params;

enum {
    B2J_FLAG_NO_PINNED = 1,  /* do not allocate pinned host staging (device-resident use only) */
    B2J_FLAG_ENCODE = 2,     /* allocate encoder state at create (else lazily on first encode) */
    B2J_FLAG_DECODE = 4      /* allocate decoder state at create (else lazily on first decode) */
};

B2J_API void b2j_default_params(b2j_params *p);
B2J_API int b2j_create(const b2j_params *p, b2j_ctx **out);
B2J_API void b2j_destroy(b2j_ctx *ctx);
B2J_API const char *b2j_last_error(const b2j_ctx *ctx);
B2J_API const char *b2j_version(void);

/* The caller's CUDA stream (cudaStream_t as void*); NULL = the context's own stream. */
/* Restart markers every `rows` MCU rows of whole-image encodes (0 = none, the default): jchuff.c emit_restart /
 * jcmarker.c emit_dri with restart_interval = rows * MCUs per row (cv2: IMWRITE_JPEG_RST_INTERVAL). */
B2J_API int b2j_set_restart_rows(b2j_ctx *ctx, int rows);
B2J_API int b2j_set_stream(b2j_ctx *ctx, void *cuda_stream);

/* Upper bound of the JPEG size b2j_encode can produce for this context. */
B2J_API size_t b2j_encode_bound(const b2j_ctx *ctx);

/* Host -> host. bgr: host pointer (pageable or pinned). out: host buffer of `cap` bytes. */
B2J_API int b2j_encode(b2j_ctx *ctx, const uint8_t *bgr, size_t step, int width, int height, uint8_t *out,
                       size_t cap, size_t *len);

/* The same in two steps, for callers that size their output after the encode (the C++ facade's std::vector):
 * b2j_encode_begin uploads and encodes (the JPEG stays in the context's device buffer) and returns its length,
 * b2j_encode_fetch copies it to host memory. */
B2J_API int b2j_encode_begin(b2j_ctx *ctx, const uint8_t *bgr, size_t step, int width, int height, size_t *len);
B2J_API int b2j_encode_fetch(b2j_ctx *ctx, uint8_t *out, size_t cap);

/* Device -> device, asynchronous on the context's stream. d_bgr: device pointer. On return *d_out points at
 * the context-owned device buffer that will hold the complete JPEG; its length is written to the device word
 * *d_len (uint64). b2j_encode_finish synchronises and returns the length. */
B2J_API int b2j_encode_device(b2j_ctx *ctx, const uint8_t *d_bgr, size_t step, int width, int height,
                              const uint8_t **d_out, const uint64_t **d_len);
B2J_API int b2j_encode_finish(b2j_ctx *ctx, size_t *len);

/* Header probe (nvjpegGetImageInfo, ImageCompressorImpl.cu:335). */
B2J_API int b2j_peek(const uint8_t *jpg, size_t len, int *width, int *height, int *css);

/* Host -> host decode to BGR interleaved. */
B2J_API int b2j_decode(b2j_ctx *ctx, const uint8_t *jpg, size_t len, uint8_t *bgr, size_t step, int *width,
                       int *height);
/* Host JPEG bytes -> device BGR (d_bgr: device pointer, pitch step); asynchronous after the header parse. */
B2J_API int b2j_decode_device(b2j_ctx *ctx, const uint8_t *jpg, size_t len, uint8_t *d_bgr, size_t step,
                              int *width, int *height);
/* A baseline JPEG whose entropy-coded segment is already in DEVICE memory: hdr = the file's bytes from SOI up to and
 * including the SOS header (host, a few hundred bytes), d_scan = the stuffed scan bytes up to the terminating marker
 * (device). height_override > 0 replaces the frame height: whole restart intervals of whole MCU rows decode as an image
 * of their own (one image decoded by several GPUs: strips.StripDecoder). Synchronous and validated.
 * d_scan may have any alignment; the de-stuffing kernel reads whole 16-byte aligned vectors, i.e. up to 15 bytes in front
 * of d_scan and behind d_scan + scan_len are read (never interpreted) -- inside the same 16-byte block of the same
 * allocation, which every CUDA allocation granule (>= 256 bytes) contains. */
B2J_API int b2j_decode_scan_device(b2j_ctx *ctx, const uint8_t *hdr, size_t hdr_len, const uint8_t *d_scan, size_t scan_len,
                                   int height_override, uint8_t *d_bgr, size_t step, int *width, int *height);
/* Reduced-size decode: libjpeg's scale_num = 1, scale_denom = denom (cv2 IMREAD_REDUCED_COLOR_denom /
 * IMREAD_REDUCED_GRAYSCALE_denom), denom in {1, 2, 4, 8}; 1 (full size) is the default. Any other value returns
 * B2J_EINVAL and leaves the setting unchanged. It applies to b2j_decode, b2j_decode_device / b2j_decode_finish and
 * b2j_decode_scan_device, for baseline, restart-marker and progressive files, on colour and gray contexts: their
 * width / height report the output size ceil(W / denom) x ceil(H / denom) (also with a NULL image, to size buffers),
 * and `step` is checked against that width. The samples equal libjpeg-turbo's DCT-scaled decode (jidctred.c, jdsample.c).
 * A context sized W x H decodes files up to that size at every scale. b2j_peek still reports the file's size; the
 * encoders, the strips, b2j_reconstruct_* and b2j_secondary* are not affected. */
B2J_API int b2j_set_decode_scale(b2j_ctx *ctx, int denom);
/* Region decode: the decodes return only columns x .. x + w - 1 and rows y .. y + h - 1 of what they would return
 * without it, in output coordinates (after the decode scale; with height_override, of the overridden image).
 * (0, 0, 0, 0), the default, is the whole image. A negative value, only one of w and h zero, or w = h = 0 with x or y
 * non-zero return B2J_EINVAL and leave the setting unchanged. It applies to b2j_decode, b2j_decode_device /
 * b2j_decode_finish and b2j_decode_scan_device: their width / height report w x h (also with a NULL image), `step` is
 * checked against w, and not one byte of the caller's image outside the w x h rectangle (pitch padding included) is
 * written. A rectangle that does not lie inside the file's output size returns B2J_EINVAL before anything runs. Only
 * the MCUs around the rectangle are transformed; in a file with restart markers only the intervals that hold them are
 * entropy-decoded. A b2j_decode_device keeps the region it was issued with until b2j_decode_finish. b2j_peek, the
 * encoders, the strips, b2j_reconstruct_* and b2j_secondary* are not affected. */
B2J_API int b2j_set_decode_region(b2j_ctx *ctx, int x, int y, int w, int h);
/* Completes the last b2j_decode_device: waits for it and validates it. The decode runs a fixed schedule of Huffman
 * synchronisation launches without asking the host; in the rare case that was too short the image is decoded again
 * here with the checked schedule. `jpg` of the b2j_decode_device call must stay valid until this returns. */
B2J_API int b2j_decode_finish(b2j_ctx *ctx);

/* Difference map and PSNR over n bytes (host pointers). */
B2J_API int b2j_diff(b2j_ctx *ctx, const uint8_t *a, const uint8_t *b, size_t n, int mode, uint8_t *out);
B2J_API int b2j_psnr(b2j_ctx *ctx, const uint8_t *a, const uint8_t *b, size_t n, double *psnr, uint64_t *ssd);
/* Same on device pointers, asynchronous; *d_ssd is a device uint64 owned by the context. */
B2J_API int b2j_diff_psnr_device(b2j_ctx *ctx, const uint8_t *d_a, const uint8_t *d_b, size_t n, int mode,
                                 uint8_t *d_out, const uint64_t **d_ssd);

/* Reconstruction without an entropy decode: the pixels every decoder produces from the LAST encode of this context,
 * from the quantised coefficients the encoder kept (set B2J_DEBUG_COEF before that encode): de-quantise + IDCT +
 * upsample + colour conversion. Device pointer, asynchronous on the context's stream. */
B2J_API int b2j_reconstruct_device(b2j_ctx *ctx, uint8_t *d_bgr, size_t step);
/* The same in two halves, for a strip of a larger image (one strip per GPU): planes first, then -- after one chroma row
 * from each neighbour strip has been copied into this strip's halo rows (row_bytes bytes each: the upper neighbour's
 * *_last rows into *_halo_top, the lower neighbour's *_first rows into *_halo_bottom) -- upsampling and colour
 * conversion; the vertical chroma filter of 4:2:0 / 4:4:0 then gives the whole image's pixels at the strip borders. */
typedef struct b2j_recon_planes {
    size_t row_bytes;                               /* true chroma width in samples */
    uint8_t *cb_first, *cr_first, *cb_last, *cr_last;            /* this strip's first / last chroma rows (device) */
    uint8_t *cb_halo_top, *cr_halo_top, *cb_halo_bottom, *cr_halo_bottom;   /* where the neighbours' rows go */
} b2j_recon_planes;
B2J_API int b2j_reconstruct_planes(b2j_ctx *ctx, b2j_recon_planes *out);
B2J_API int b2j_reconstruct_color(b2j_ctx *ctx, uint8_t *d_bgr, size_t step, int halo_top, int halo_bottom);

/* Secondary compression, device resident (README.md:8): encode -> reconstruct (from the encoder's coefficients, no
 * Huffman decode, no host round trip) -> difference map + SSD -> encode(difference). d_bgr: device pointer, contiguous
 * rows (step == width * 3). Asynchronous; the returned pointers are context-owned device buffers (primary JPEG,
 * secondary JPEG, reconstruction, difference map; any may be NULL). b2j_secondary_finish waits, validates both
 * encodes and returns the two lengths, PSNR(orig, recon) and the exact SSD. */
B2J_API int b2j_secondary_device(b2j_ctx *ctx, const uint8_t *d_bgr, size_t step, int width, int height, int diff_mode,
                                 const uint8_t **d_jpg1, const uint8_t **d_jpg2, const uint8_t **d_recon,
                                 const uint8_t **d_diff);
B2J_API int b2j_secondary_finish(b2j_ctx *ctx, size_t *len1, size_t *len2, double *psnr, uint64_t *ssd);

/* Results of the last b2j_secondary_device + _finish (or b2j_secondary) -> host memory; any pointer may be NULL. */
B2J_API int b2j_secondary_fetch(b2j_ctx *ctx, uint8_t *jpg1, size_t cap1, uint8_t *jpg2, size_t cap2, uint8_t *recon,
                                size_t recon_step);

/* The same from and to host memory (upload, b2j_secondary_device, downloads). Any output pointer may be NULL. */
B2J_API int b2j_secondary(b2j_ctx *ctx, const uint8_t *bgr, size_t step, int width, int height, int diff_mode,
                          uint8_t *jpg1, size_t cap1, size_t *len1, uint8_t *jpg2, size_t cap2, size_t *len2,
                          uint8_t *recon, size_t recon_step, double *psnr);

/* ---- staged (strip) interface used by the multi-GPU host: one MCU-row strip per context/GPU -------------
 * phase1: colour/downsample/FDCT/quant (+ symbol histograms when optimize) of a device-resident strip.
 * Between phases the host runs the collectives on the device words exposed by b2j_strip_state. */
typedef struct b2j_strip_state {
    uint32_t *d_hist;       /* [4][257] symbol counts: DC0, AC0, DC1, AC1 (allreduce SUM target) */
    int16_t *d_last_dc;     /* [3] quantised DC of the strip's last Y, Cb, Cr blocks (allgather source) */
    int16_t *d_pred_in;     /* [3] DC predictors at the strip start (host fills from the previous rank) */
    uint64_t *d_strip_bits; /* [2]: entropy bits of this strip (unstuffed), first 32 bits of its bit string */
    uint64_t *d_out_len;    /* bytes this strip produced in d_out (header included on first strip) */
    uint8_t *d_out;
    void *d_record;         /* b2j_strip_record of this strip (one-collective schedule: allgather source) */
} b2j_strip_state;

B2J_API int b2j_strip_state_get(b2j_ctx *ctx, b2j_strip_state *st);
B2J_API int b2j_strip_phase1(b2j_ctx *ctx, const uint8_t *d_bgr, size_t step, int width, int rows);
/* DC-difference symbols at the strip start need d_pred_in: counted here, after the last-DC exchange. */
B2J_API int b2j_strip_phase1b(b2j_ctx *ctx);
/* tables from d_hist (after allreduce) + entropy-code the strip at bit phase 0 */
B2J_API int b2j_strip_phase2(b2j_ctx *ctx, int full_width, int full_height);
/* shift to the global bit phase, byte-stuff. skip_bits = (8 - global_start_bit%8)%8, ext_byte = next strip's
 * first 8 bits (0xFF for the last strip). flags: bit0 = emit headers first, bit1 = append EOI. */
B2J_API int b2j_strip_phase3(b2j_ctx *ctx, int skip_bits, int ext_byte, int flags);
/* Same, with the seam derived on the device (no host synchronisation in the multi-GPU step): d_bits_all is the
 * all-gathered table [world][2] of int64 {d_strip_bits[0], d_strip_bits[1]} of every strip, in strip order. */
B2J_API int b2j_strip_phase3_dev(b2j_ctx *ctx, const int64_t *d_bits_all, int rank, int world, int flags);

/* One-collective schedule (what StripEncoder uses on GPUs): phase1x, ONE allgather of the strips' records, phase2x.
 * The record carries the strip's symbol counts (always taken), its first/last DCs and its first tokens; with all
 * records every rank derives the image histogram, the DC symbols at the strip starts, every strip's entropy bit
 * count (histogram x code lengths: the bit phase of a strip does not wait for the other strips' entropy coders) and
 * the bits that complete its last byte. phase2x = tables + entropy coding + seam + byte stuffing of this strip;
 * the predicted bit count is checked against the coded one on the device (b2j_encode_finish reports a mismatch). */
#define B2J_STRIP_RECORD_BYTES 4176
typedef struct b2j_strip_record {
    uint32_t hist[4 * 257]; /* DC0, AC0, DC1, AC1; the DC symbols of the strip's first MCU are not included */
    int16_t first_dc[4];    /* quantised DC of the strip's first Y, Cb, Cr blocks */
    int16_t last_dc[4];     /* ... of its last Y, Cb, Cr blocks */
    uint32_t tok[8];        /* first entropy tokens of the strip (engine-internal format) */
    uint32_t ntok;
    uint32_t pad[3];
} b2j_strip_record;
/* Peer-memory variant (GPUs of one node with P2P access, one process per GPU): no collective at all. Set-up, once:
 * every rank calls b2j_peer_export (allocates its arena, returns a 64-byte cudaIpcMemHandle_t), the host exchanges the
 * handles, each rank maps the others' with b2j_peer_open and calls b2j_peer_connect(rank, world, arenas[world])
 * (arenas[rank] is ignored), then a host barrier. From then on b2j_strip_phase1x also stores the record into every
 * rank's arena over NVLink and raises a flag there, and b2j_strip_phase2x(ctx, NULL, ...) waits (bounded: error 9 after
 * B2J_PEER_TIMEOUT_MS, default 10 s, never a hang) for the world's flags of this image before merging. All ranks must encode the same number of
 * images. Same-process callers (tests) pass raw arena pointers from b2j_peer_export to b2j_peer_connect. */
B2J_API int b2j_peer_export(b2j_ctx *ctx, void *ipc_handle_64, void **d_arena);
B2J_API int b2j_peer_open(b2j_ctx *ctx, const void *ipc_handle_64, void **d_ptr);
B2J_API int b2j_peer_connect(b2j_ctx *ctx, int rank, int world, void *const *d_arenas);
B2J_API int b2j_strip_phase1x(b2j_ctx *ctx, const uint8_t *d_bgr, size_t step, int width, int rows);
B2J_API int b2j_strip_phase2x(b2j_ctx *ctx, const void *d_records_all, int rank, int world, int full_width,
                              int full_height, int flags);

/* ---- several GPUs of one node from ONE process and one host thread (SURVEY.md 8b: ngpus / device_ids) -------------
 * One image is cut into MCU-row strips, one per GPU; the strips exchange their 4 KB records through peer memory
 * (NVLink stores + flags, no collective), every strip's rows go up over its own GPU's link in groups with the fdct of
 * a group behind it, every strip's bytes come down straight to their place in `out`. The stream is byte for byte the
 * single-GPU stream. device_ids == NULL: devices 0 .. ngpus-1 (at most 16). */
typedef struct b2j_multi b2j_multi;
B2J_API int b2j_multi_create(const b2j_params *p, int ngpus, const int *device_ids, b2j_multi **out);
B2J_API void b2j_multi_destroy(b2j_multi *m);
B2J_API int b2j_multi_encode(b2j_multi *m, const uint8_t *bgr, size_t step, int width, int height, uint8_t *out,
                             size_t cap, size_t *len);
/* in two steps (the caller sizes its buffer to the stream): encode on every GPU, then fetch the strips' bytes */
B2J_API int b2j_multi_encode_begin(b2j_multi *m, const uint8_t *bgr, size_t step, int width, int height, size_t *len);
B2J_API int b2j_multi_encode_fetch(b2j_multi *m, uint8_t *out, size_t cap);
B2J_API const char *b2j_multi_last_error(const b2j_multi *m);

/* ---- introspection used by the parity tests (device -> host copies of intermediate state) ------------- */
enum { B2J_DBG_COEF = 0, B2J_DBG_HIST = 1, B2J_DBG_TABLES = 2, B2J_DBG_TILE_BITS = 3, B2J_DBG_DEC_COEF = 4,
       B2J_DBG_TOKEN_COUNT = 5, B2J_DBG_TOKENS = 6, B2J_DBG_TILE_RECS = 7, B2J_DBG_SLOTS = 8 /* SLOTS: the per-tile bit buffers (SLOT_WORDS = 13312 uint32 per tile, MSB first). TOKENS: the token pool (uint32 each, csrc/common.cuh); TILE_RECS: one 24-byte record per fdct tile. DEC_COEF: decoded blocks, zig-zag order, DC as difference. TOKEN_COUNT: uint32: run-length tokens of the last encode (4 bytes each between the two passes) */ };
B2J_API int b2j_debug_read(b2j_ctx *ctx, int what, void *dst, size_t cap, size_t *len);
/* flags bit0 (B2J_DEBUG_COEF): the next encodes also store the quantised coefficients for B2J_DBG_COEF */
/* bit1 (B2J_DEBUG_SMALL_PACK_BUFFERS): the entropy coder's per-warp bit buffers overflow on purpose (tests its
 * two-pass recovery path); output is unchanged */
/* bit2 (B2J_DEBUG_SHORT_DECODE_SCHEDULE): the decoder's unchecked synchronisation schedule is cut to one launch, so
 * every multi-chunk image takes the validated retry; output is unchanged */
/* bit3: unused and ignored; older callers may still set it, so it must not be given a new meaning */
enum { B2J_DEBUG_COEF = 1, B2J_DEBUG_SMALL_PACK_BUFFERS = 2, B2J_DEBUG_SHORT_DECODE_SCHEDULE = 4 };
B2J_API int b2j_set_debug(b2j_ctx *ctx, int flags);

/* per-stage device times (ms) of the last encode/decode, measured with CUDA events on the context stream */
typedef struct b2j_timings {
    float h2d, fdct, hist_edge, tables, pack, scan, stuff, d2h, total;
    float dec_parse, dec_sync, dec_write, dec_idct, dec_color;
} b2j_timings;
B2J_API int b2j_last_timings(b2j_ctx *ctx, b2j_timings *t);
B2J_API int b2j_enable_timing(b2j_ctx *ctx, int on);

/* number of kernels this library launched since the context was created */
B2J_API uint64_t b2j_launch_count(const b2j_ctx *ctx);

/* pinned host memory helpers for callers that want zero-copy-staged uploads */
B2J_API void *b2j_host_alloc(size_t bytes);
B2J_API void b2j_host_free(void *p);

#ifdef __cplusplus
}
#endif
#endif /* B2JPEG_H_ */
