// api.cu -- the extern "C" boundary of libb2jpeg.so (include/b2jpeg.h): context, device buffers, stage sequencing.
// Host-side mirror of NvjpegCompressRunnerImpl (reference src/ImageCompressorDll/ImageCompressorImpl.cu:19-117
// env setup/teardown, :269-294 CompressWorker, :311-385 DecodeWorker) with nvJPEG replaced by this library's kernels.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <new>
#include <vector>

#include "../../include/b2jpeg.h"
#include "common.cuh"
#include "dec.h"
#include "dec_kernels.h"
#include "hostpipe.h"
#include "kernels.h"

using namespace b2j;

namespace {

struct Ctrl {  // zeroed before every encode with one memset
    union {
        uint32_t hist[4 * 257];
        StripRecord rec;   // the strip exchange record starts with the histogram
    };
    uint32_t ticket;
    uint32_t pool_count;
    uint32_t scan_ticket;
    uint32_t pad0;
    // ---- fetched by the host in one copy (same layout as HostRet)
    uint64_t out_len;
    uint64_t strip_bits[2];
    uint64_t ssd;
    uint32_t err;        // k_stuff / look-backs
    uint32_t huff_err;   // k_tables
    // ----
    int seam[2];         // [0] skip bits, [1] ext byte XOR 0xFF (so that all-zero means "whole image": skip 0, pad with ones)
};

struct HostRet {  // pinned
    uint64_t out_len;
    uint64_t strip_bits[2];
    uint64_t ssd;
    uint32_t err;
    uint32_t huff_err;
};

}  // namespace

struct b2j_ctx {
    b2j_params p;
    int device;
    cudaStream_t own_stream, copy_stream, stream;
    Geom cap_g;  // geometry of the configured (maximum) image
    Geom g;      // geometry of the current image / strip
    QuantDev hq;
    // encoder state
    bool enc_ready;
    uint8_t *d_img;
    size_t d_img_bytes;
    int16_t *d_coef;      // only with B2J_DEBUG_COEF
    uint32_t *d_pool;     // token pool, 64 tokens per block worst case
    TileRec *d_recs;
    int tiles_cap;
    size_t slot_words_cap;
    int debug;
    uint32_t *d_slots, *d_tile_bits;
    uint64_t *d_tile_off, *d_desc, *d_sdesc;   // look-back descriptors: byte stuffing, tile scan
    uint32_t *d_chunk_tile;                    // [ndesc] tile holding the first bit of every k_stuff chunk (written by the scan)
    size_t ndesc, nsdesc;
    Ctrl *d_ctrl;
    int16_t *d_pred_in;
    HuffDev *d_huff;
    QuantDev *d_quant;
    uint8_t *d_out;
    size_t out_cap;
    HostRet *h_ret;
    cudaEvent_t ev[12], ev_copy[64];
    bool timing;
    b2j_timings tm;
    uint64_t launches;
    char err[256];
    // decoder + secondary state
    b2j::Decoder *dec;
    uint8_t *d_recon, *d_diff;
    size_t d_recon_bytes, d_diff_bytes;
    // pageable host buffers: copy threads + pinned staging ring (hostpipe.h), created on first use
    b2j::CopyPool *pool;
    b2j::StageRing ring;
    // last b2j_decode_device call (for b2j_decode_finish)
    const uint8_t *last_jpg;
    size_t last_len, last_step;
    uint8_t *last_bgr;
    int last_scale;                // ... and the scale it was issued with (its checked retry keeps it)
    int dec_scale;                 // decode output at 1 / dec_scale (1, 2, 4, 8); b2j_set_decode_scale
    b2j_ctx *second;  // encoder for the difference image (secondary compression)
    uint8_t *d_rplanes; size_t rplanes_bytes;   // reconstruction from the encoder's coefficients: sample planes
    void *d_rtb;                                // ... and de-quantisation tables (a DecTables with q filled)
    // peer-memory exchange of the strip records (multi-GPU encode without a collective)
    XchgArena *d_arena;            // this rank's arena (peers store into it)
    XchgArena **d_peers;           // device array [peer_world] of every rank's arena
    void *peer_opened[XCHG_MAX_WORLD];   // mappings from b2j_peer_open (closed in b2j_destroy)
    int n_opened, peer_rank, peer_world;
    int rst_rows;                  // restart interval in MCU rows (0: none); b2j_set_restart_rows
    size_t sec_pixels;             // b2j_secondary_device: samples of the image in flight (PSNR denominator)
    uint32_t xseq;                 // images exchanged so far (identical on every rank)
    unsigned long long peer_timeout_ns;   // bound of the wait for the peers' records (B2J_PEER_TIMEOUT_MS, default 10 s)
};

extern "C" { static int upload_linear(void *user, uint8_t *d_dst, const uint8_t *src, size_t n, cudaStream_t s); }

#define CK(call)                                                                                        \
    do {                                                                                                \
        cudaError_t _e = (call);                                                                        \
        if (_e != cudaSuccess) {                                                                        \
            snprintf(ctx->err, sizeof(ctx->err), "%s at %s:%d", cudaGetErrorString(_e), __FILE__, __LINE__); \
            return B2J_ECUDA;                                                                           \
        }                                                                                               \
    } while (0)

// B2J_CSS_GRAY: one component, one block per MCU (nc = 1, bpm = 1, hs = vs = 1); component 0 only in wib/hib/dw/dh
static int make_geom(int W, int H, int css, Geom *g) {
    static const int HS[5] = {1, 2, 1, 2, 4}, VS[5] = {1, 1, 2, 2, 1};
    const bool gray = css == B2J_CSS_GRAY;
    if (W <= 0 || H <= 0 || W > 65535 || H > 65535 || css < 0 || (css > 4 && !gray)) return B2J_EINVAL;
    memset(g, 0, sizeof(*g));
    g->W = W; g->H = H; g->hs = gray ? 1 : HS[css]; g->vs = gray ? 1 : VS[css];
    g->nc = gray ? 1 : 3;
    g->mcux = (W + 8 * g->hs - 1) / (8 * g->hs);
    g->mcuy = (H + 8 * g->vs - 1) / (8 * g->vs);
    g->bpm = gray ? 1 : g->hs * g->vs + 2;
    for (int c = 0; c < g->nc; c++) {
        const int h = c ? 1 : g->hs, v = c ? 1 : g->vs;
        g->dw[c] = (W * h + g->hs - 1) / g->hs;
        g->dh[c] = (H * v + g->vs - 1) / g->vs;
        g->wib[c] = (g->dw[c] + 7) / 8;
        g->hib[c] = (g->dh[c] + 7) / 8;
    }
    const long long nb = (long long)g->mcux * g->mcuy * g->bpm;
    if (nb > 0x7fffffffLL / 64) return B2J_EINVAL;
    g->nblocks = (int)nb;
    // fdct tiles: as even as possible, an even MCU count per tile (16-byte alignment of the bulk copies)
    const int tmax = fdct_tm_max(g->hs, g->vs, g->nc);
    g->tiles_x = (g->mcux + tmax - 1) / tmax;
    int tm = (g->mcux + g->tiles_x - 1) / g->tiles_x;
    tm = (tm + 1) & ~1;
    if (tm > tmax) tm = tmax;
    g->tm = tm;
    g->tiles_x = (g->mcux + tm - 1) / tm;
    g->ntiles = g->tiles_x * g->mcuy;
    return B2J_OK;
}

// jcparam.c jpeg_set_quality + exact reciprocals for the forward quantiser
static void make_quant(int quality, QuantDev *q) {
    static const uint8_t L[64] = {16, 11, 10, 16, 24,  40,  51,  61,  12, 12, 14, 19, 26,  58,  60,  55,
                                  14, 13, 16, 24, 40,  57,  69,  56,  14, 17, 22, 29, 51,  87,  80,  62,
                                  18, 22, 37, 56, 68,  109, 103, 77,  24, 35, 55, 64, 81,  104, 113, 92,
                                  49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99};
    static const uint8_t Cq[64] = {17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99, 24, 26, 56, 99, 99, 99,
                                   99, 99, 47, 66, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99,
                                   99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99};
    int ql = quality < 1 ? 1 : (quality > 100 ? 100 : quality);
    const int scale = ql < 50 ? 5000 / ql : 200 - 2 * ql;
    for (int t = 0; t < 2; t++)
        for (int i = 0; i < 64; i++) {
            long v = ((long)(t ? Cq[i] : L[i]) * scale + 50) / 100;
            if (v < 1) v = 1;
            if (v > 255) v = 255;
            const uint32_t d = 8u * (uint32_t)v;
            q->q[t][i] = (uint16_t)v;
            q->finv[t][i] = (float)((1.0 / (double)d) * (1.0 + 1.0 / 1048576.0)) * 4096.0f;   // see k_fdct: exact for |c| <= 2^18
        }
}

// bytes per pixel of the context's images: 1 (8-bit gray) or 3 (BGR)
static inline int chans(const b2j_ctx *ctx) { return ctx->p.css == B2J_CSS_GRAY ? 1 : 3; }

// the entry points that assume three components (strips, peers, reconstruction, secondary compression) refuse gray
static int refuse_gray(b2j_ctx *ctx, const char *what) {
    if (ctx->p.css != B2J_CSS_GRAY) return B2J_OK;
    snprintf(ctx->err, sizeof(ctx->err), "%s: not supported on a gray (B2J_CSS_GRAY) context", what);
    return B2J_EINVAL;
}
#define REFUSE_GRAY(ctx, what) do { const int _r = refuse_gray((ctx), (what)); if (_r) return _r; } while (0)

extern "C" {

void b2j_default_params(b2j_params *p) {
    p->width = 8320; p->height = 40000; p->quality = 95; p->optimize = 1; p->css = B2J_CSS_422; p->device = -1; p->flags = 0;
}

const char *b2j_version(void) { return "b2jpeg 0.1 (sm_100a)"; }

const char *b2j_last_error(const b2j_ctx *ctx) { return ctx ? ctx->err : "null context"; }

static int ensure_tiles(b2j_ctx *ctx, const Geom &g) {
    if (g.ntiles <= ctx->tiles_cap) return B2J_OK;
    cudaFree(ctx->d_slots); cudaFree(ctx->d_tile_bits); cudaFree(ctx->d_tile_off); cudaFree(ctx->d_recs);
    ctx->d_slots = nullptr; ctx->d_tile_bits = nullptr; ctx->d_tile_off = nullptr; ctx->d_recs = nullptr; ctx->tiles_cap = 0;
    const int n = g.ntiles + g.ntiles / 8 + 16;
    const bool was_ready = ctx->enc_ready;
    ctx->enc_ready = false;   // stays false if an allocation below fails: no phase launches with null tile buffers
    CK(cudaMalloc(&ctx->d_slots, (size_t)n * SLOT_WORDS * 4));
    CK(cudaMalloc(&ctx->d_tile_bits, (size_t)(n + 1) * 4));
    CK(cudaMalloc(&ctx->d_tile_off, (size_t)(n + 2) * 8));
    CK(cudaMalloc(&ctx->d_recs, (size_t)(n + 1) * sizeof(TileRec)));
    ctx->tiles_cap = n;
    ctx->enc_ready = was_ready;
    return B2J_OK;
}

// Everything an encode needs zeroed lives in ONE allocation, cleared by one memset per image:
// [Ctrl | pred_in (16 B) | tile-scan descriptors (nsdesc) | byte-stuffing descriptors (ndesc, used prefix cleared)]
constexpr size_t ARENA_CTRL = (sizeof(Ctrl) + 15) & ~(size_t)15;
static int alloc_zero_arena(b2j_ctx *ctx, size_t nsdesc) {
    if (ctx->d_ctrl) { cudaFree(ctx->d_ctrl); ctx->d_ctrl = nullptr; }
    ctx->nsdesc = nsdesc;
    uint8_t *p = nullptr;
    CK(cudaMalloc(&p, ARENA_CTRL + 16 + (ctx->nsdesc + ctx->ndesc) * 8));
    ctx->d_ctrl = reinterpret_cast<Ctrl *>(p);
    ctx->d_pred_in = reinterpret_cast<int16_t *>(p + ARENA_CTRL);
    ctx->d_sdesc = reinterpret_cast<uint64_t *>(p + ARENA_CTRL + 16);
    ctx->d_desc = ctx->d_sdesc + ctx->nsdesc;
    return B2J_OK;
}

static int enc_alloc(b2j_ctx *ctx) {
    if (ctx->enc_ready) return B2J_OK;
    const Geom &g = ctx->cap_g;
    // every buffer is allocated only while its pointer is null: a call that failed half way can be repeated
    if (!ctx->d_pool) CK(cudaMalloc(&ctx->d_pool, (size_t)g.nblocks * 64 * 4 + 64));  // +64: k_pack reads whole 16-byte groups
    int rc = ensure_tiles(ctx, g); if (rc) return rc;
    ctx->out_cap = (size_t)g.nblocks * 208 + 4096 + (size_t)g.mcuy * 3;   // + pad/RSTn bytes of restart intervals
    if (!ctx->d_out) CK(cudaMalloc(&ctx->d_out, ctx->out_cap));
    ctx->ndesc = ctx->out_cap / STUFF_CHUNK + 4;
    // 1024 scan descriptors cover 4M tiles: no geometry within the configured size re-allocates (b2j_strip_state
    // hands out pointers into this arena)
    if (!ctx->d_ctrl) { rc = alloc_zero_arena(ctx, std::max<size_t>((size_t)scan_desc_count(g.ntiles) + 64, 1024)); if (rc) return rc; }
    if (!ctx->d_chunk_tile) CK(cudaMalloc(&ctx->d_chunk_tile, ctx->ndesc * 4));
    if (!ctx->d_huff) CK(cudaMalloc(&ctx->d_huff, sizeof(HuffDev)));
    if (!ctx->d_quant) CK(cudaMalloc(&ctx->d_quant, sizeof(QuantDev)));
    CK(cudaMemcpy(ctx->d_quant, &ctx->hq, sizeof(QuantDev), cudaMemcpyHostToDevice));
    ctx->enc_ready = true;
    return B2J_OK;
}

static int ensure_debug(b2j_ctx *ctx) {
    if ((ctx->debug & 1) && !ctx->d_coef) CK(cudaMalloc(&ctx->d_coef, (size_t)ctx->cap_g.nblocks * 128));
    return B2J_OK;
}

int b2j_create(const b2j_params *p, b2j_ctx **out) {
    if (!p || !out) return B2J_EINVAL;
    b2j_ctx *ctx = new (std::nothrow) b2j_ctx();
    if (!ctx) return B2J_ENOMEM;
    memset(ctx, 0, sizeof(*ctx));
    ctx->p = *p;
    int rc = make_geom(p->width, p->height, p->css, &ctx->cap_g);
    if (rc) { delete ctx; return rc; }
    ctx->g = ctx->cap_g;
    ctx->dec_scale = 1;
    make_quant(p->quality, &ctx->hq);
    cudaError_t e;
    if (p->device >= 0) {
        e = cudaSetDevice(p->device);
        if (e != cudaSuccess) { delete ctx; return B2J_ECUDA; }
    }
    e = cudaGetDevice(&ctx->device);
    if (e != cudaSuccess) { delete ctx; return B2J_ECUDA; }  // no CUDA device: fail loudly, there is no CPU path
    if (cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking) != cudaSuccess) { b2j_destroy(ctx); return B2J_ECUDA; }
    ctx->stream = ctx->own_stream;
    for (auto &ev : ctx->ev) cudaEventCreate(&ev);
    for (auto &ev : ctx->ev_copy) cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
    if (cudaHostAlloc(&ctx->h_ret, sizeof(HostRet), cudaHostAllocDefault) != cudaSuccess) { b2j_destroy(ctx); return B2J_ECUDA; }
    *out = ctx;
    if (p->flags & B2J_FLAG_ENCODE) { rc = enc_alloc(ctx); if (rc) { b2j_destroy(ctx); *out = nullptr; return rc; } }
    return B2J_OK;
}

void b2j_destroy(b2j_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    if (ctx->second) b2j_destroy(ctx->second);
    if (ctx->dec) dec_destroy(ctx->dec);
    delete ctx->pool;
    ctx->ring.release();
    cudaFree(ctx->d_img); cudaFree(ctx->d_coef); cudaFree(ctx->d_pool); cudaFree(ctx->d_recs); cudaFree(ctx->d_slots); cudaFree(ctx->d_tile_bits);
    for (int i = 0; i < ctx->n_opened; i++) cudaIpcCloseMemHandle(ctx->peer_opened[i]);
    cudaFree(ctx->d_arena); cudaFree(ctx->d_peers);
    cudaFree(ctx->d_chunk_tile);
    cudaFree(ctx->d_tile_off); cudaFree(ctx->d_ctrl);   // d_pred_in, d_sdesc, d_desc live in d_ctrl's allocation
    cudaFree(ctx->d_huff); cudaFree(ctx->d_quant); cudaFree(ctx->d_out); cudaFree(ctx->d_recon); cudaFree(ctx->d_diff);
    cudaFree(ctx->d_rplanes); cudaFree(ctx->d_rtb);
    if (ctx->h_ret) cudaFreeHost(ctx->h_ret);
    for (auto &ev : ctx->ev) if (ev) cudaEventDestroy(ev);
    for (auto &ev : ctx->ev_copy) if (ev) cudaEventDestroy(ev);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    delete ctx;
}

int b2j_set_stream(b2j_ctx *ctx, void *s) {
    if (!ctx) return B2J_EINVAL;
    ctx->stream = s ? (cudaStream_t)s : ctx->own_stream;
    return B2J_OK;
}

size_t b2j_encode_bound(const b2j_ctx *ctx) { return ctx ? (size_t)ctx->cap_g.nblocks * 208 + 4096 + (size_t)ctx->cap_g.mcuy * 3 : 0; }

// Restart markers every `rows` MCU rows (0 = none): DRI = rows * MCUs per row in the header, RSTn between the intervals,
// DC predictors restart (jchuff.c emit_restart; the stream equals libjpeg-turbo's with restart_interval = rows * mcux).
// Whole-image encodes only; the interval must fit DRI's 16 bits for the configured width.
int b2j_set_restart_rows(b2j_ctx *ctx, int rows) {
    if (!ctx || rows < 0 || (long long)rows * ctx->cap_g.mcux > 65535) return B2J_EINVAL;
    ctx->rst_rows = rows;
    return B2J_OK;
}
// Reduced-size decode: libjpeg's scale_num = 1, scale_denom = denom (cv2 IMREAD_REDUCED_*_denom). The entropy stages are
// unchanged; the back end runs jidctred.c's smaller inverse DCTs (dec_scaled.cu).
int b2j_set_decode_scale(b2j_ctx *ctx, int denom) {
    if (!ctx || (denom != 1 && denom != 2 && denom != 4 && denom != 8)) return B2J_EINVAL;
    ctx->dec_scale = denom;
    return B2J_OK;
}
uint64_t b2j_launch_count(const b2j_ctx *ctx) { return ctx ? ctx->launches : 0; }
int b2j_set_debug(b2j_ctx *ctx, int flags) { if (!ctx) return B2J_EINVAL; ctx->debug = flags; return B2J_OK; }
int b2j_enable_timing(b2j_ctx *ctx, int on) { if (!ctx) return B2J_EINVAL; ctx->timing = on != 0; return B2J_OK; }

void *b2j_host_alloc(size_t bytes) { void *p = nullptr; return cudaHostAlloc(&p, bytes, cudaHostAllocDefault) == cudaSuccess ? p : nullptr; }
void b2j_host_free(void *p) { if (p) cudaFreeHost(p); }

// ------------------------------------------------------------------------------------------ staged encode
static int set_strip_geom(b2j_ctx *ctx, int width, int rows) {
    Geom g;
    int rc = make_geom(width, rows, ctx->p.css, &g);
    if (rc) return rc;
    if (g.nblocks > ctx->cap_g.nblocks) { snprintf(ctx->err, sizeof(ctx->err), "image %dx%d exceeds the context's %dx%d", width, rows, ctx->p.width, ctx->p.height); return B2J_ESIZE; }
    ctx->g = g;
    rc = ensure_tiles(ctx, g); if (rc) return rc;
    return ensure_debug(ctx);
}

static int enc_reset(b2j_ctx *ctx) {   // also zeroes pred_in: strip hosts fill it AFTER phase1
    if ((size_t)scan_desc_count(ctx->g.ntiles) > ctx->nsdesc) {   // strips with more (smaller) tiles than the configured image
        CK(cudaStreamSynchronize(ctx->stream));
        int rc = alloc_zero_arena(ctx, (size_t)scan_desc_count(ctx->g.ntiles) + 64); if (rc) return rc;
    }
    // descriptors actually reachable for this image: bounded by its worst-case entropy bytes
    size_t nd = std::min(ctx->ndesc, ((size_t)ctx->g.nblocks * 208) / STUFF_CHUNK + 4);
    CK(cudaMemsetAsync(ctx->d_ctrl, 0, ARENA_CTRL + 16 + (ctx->nsdesc + nd) * 8, ctx->stream));
    return B2J_OK;
}

static inline void tick(b2j_ctx *ctx, int i) { if (ctx->timing) cudaEventRecord(ctx->ev[i], ctx->stream); }

int b2j_strip_phase1(b2j_ctx *ctx, const uint8_t *d_bgr, size_t step, int width, int rows) {
    if (!ctx || !d_bgr) return B2J_EINVAL;
    REFUSE_GRAY(ctx, "b2j_strip_phase1");
    CK(cudaSetDevice(ctx->device));
    int rc = enc_alloc(ctx); if (rc) return rc;
    rc = set_strip_geom(ctx, width, rows); if (rc) return rc;
    rc = enc_reset(ctx); if (rc) return rc;
    tick(ctx, 1);
    CK(launch_fdct(d_bgr, step, ctx->g, ctx->d_quant, ctx->d_pool, &ctx->d_ctrl->pool_count, ctx->d_recs, ctx->d_ctrl->hist, ctx->p.optimize, 0, ctx->g.mcuy, (ctx->debug & 1) ? ctx->d_coef : nullptr, ctx->stream));
    CK(launch_dc_edge_hist(ctx->d_recs, ctx->g, ctx->d_pred_in, ctx->d_ctrl->hist, ctx->d_ctrl->rec.last_dc, 0, ctx->d_pool, 0, nullptr, 0, ctx->stream));
    ctx->launches += 2;
    tick(ctx, 2);
    return B2J_OK;
}

// phase1b / phase2 / phase3: the whole-image encode's back half on every context; the exported strip entry points
// below wrap them and refuse gray contexts
static int strip_phase1b(b2j_ctx *ctx) {
    if (!ctx || !ctx->enc_ready) return B2J_EINVAL;
    CK(cudaSetDevice(ctx->device));
    CK(launch_dc_edge_hist(ctx->d_recs, ctx->g, ctx->d_pred_in, ctx->d_ctrl->hist, ctx->d_ctrl->rec.last_dc, ctx->p.optimize, ctx->d_pool, 1, nullptr, ctx->rst_rows * ctx->g.tiles_x, ctx->stream));
    ctx->launches += 1;
    tick(ctx, 3);
    return B2J_OK;
}

static int strip_phase2(b2j_ctx *ctx, int full_w, int full_h) {
    if (!ctx || !ctx->enc_ready) return B2J_EINVAL;
    CK(cudaSetDevice(ctx->device));
    // header is always composed; phase3 decides whether it is part of this strip's output (hdr_len is re-set there)
    CK(launch_tables(ctx->d_ctrl->hist, ctx->p.optimize, ctx->d_huff, ctx->d_quant, full_w, full_h, ctx->g.hs, ctx->g.vs, ctx->g.nc, ctx->d_out, 1, ctx->rst_rows * ctx->g.mcux, &ctx->d_ctrl->huff_err, ctx->stream));
    tick(ctx, 4);
    CK(launch_pack(ctx->d_pool, ctx->d_recs, ctx->g, ctx->d_huff, ctx->d_slots, ctx->d_tile_bits, ctx->debug & 2, ctx->stream));
    if (ctx->rst_rows) {   // pad every interval to a byte boundary and append its RSTn marker, before the tile scan
        CK(launch_rst_pad(ctx->d_slots, ctx->d_tile_bits, ctx->g.ntiles, ctx->rst_rows * ctx->g.tiles_x, ctx->stream));
        ctx->launches += 1;
    }
    tick(ctx, 5);
    CK(launch_scan_tiles(ctx->d_tile_bits, ctx->g.ntiles, ctx->d_tile_off, ctx->d_slots, ctx->d_ctrl->strip_bits, ctx->d_sdesc,
                         &ctx->d_ctrl->scan_ticket, ctx->d_chunk_tile, (uint32_t)ctx->ndesc, &ctx->d_ctrl->err, ctx->stream));
    ctx->launches += 3;
    tick(ctx, 6);
    return B2J_OK;
}

__global__ void k_set_hdr_len(HuffDev *h, uint32_t v) { h->hdr_len = v; }

static int phase3_launch(b2j_ctx *ctx, int flags, bool hdr_done = false) {
    if (!(flags & 1) && !hdr_done) { k_set_hdr_len<<<1, 1, 0, ctx->stream>>>(ctx->d_huff, 0); ctx->launches++; }
    StuffArgs a;
    a.slots = ctx->d_slots; a.tile_bits = ctx->d_tile_bits; a.tile_off = ctx->d_tile_off; a.ntiles = ctx->g.ntiles;
    a.chunk_tile = ctx->d_chunk_tile;
    a.rst_tiles = ctx->rst_rows * ctx->g.tiles_x;
    a.seam = ctx->d_ctrl->seam; a.append_eoi = (flags & 2) ? 1 : 0; a.huff = ctx->d_huff;
    a.out = ctx->d_out; a.cap = ctx->out_cap; a.desc = ctx->d_desc; a.ticket = &ctx->d_ctrl->ticket;
    a.out_len = &ctx->d_ctrl->out_len; a.err = &ctx->d_ctrl->err;
    CK(launch_stuff(a, 148 * STUFF_CTAS, ctx->stream));
    ctx->launches += 1;
    tick(ctx, 7);
    return B2J_OK;
}

static int strip_phase3(b2j_ctx *ctx, int skip_bits, int ext_byte, int flags) {
    if (!ctx || !ctx->enc_ready || skip_bits < 0 || skip_bits > 7) return B2J_EINVAL;
    CK(cudaSetDevice(ctx->device));
    if (skip_bits != 0 || (ext_byte & 0xFF) != 0xFF) {   // the zeroed control block already says "skip 0, pad with ones"
        CK(launch_set_seam(ctx->d_ctrl->seam, skip_bits, ext_byte & 0xFF, ctx->stream));
        ctx->launches += 1;
    }
    return phase3_launch(ctx, flags);
}

int b2j_strip_phase1b(b2j_ctx *ctx) {
    if (ctx) REFUSE_GRAY(ctx, "b2j_strip_phase1b");
    return strip_phase1b(ctx);
}
int b2j_strip_phase2(b2j_ctx *ctx, int full_w, int full_h) {
    if (ctx) REFUSE_GRAY(ctx, "b2j_strip_phase2");
    return strip_phase2(ctx, full_w, full_h);
}
int b2j_strip_phase3(b2j_ctx *ctx, int skip_bits, int ext_byte, int flags) {
    if (ctx) REFUSE_GRAY(ctx, "b2j_strip_phase3");
    return strip_phase3(ctx, skip_bits, ext_byte, flags);
}

int b2j_strip_phase3_dev(b2j_ctx *ctx, const int64_t *d_bits_all, int rank, int world, int flags) {
    if (!ctx || !ctx->enc_ready || !d_bits_all || rank < 0 || rank >= world) return B2J_EINVAL;
    REFUSE_GRAY(ctx, "b2j_strip_phase3_dev");
    CK(cudaSetDevice(ctx->device));
    CK(launch_seam_from_bits(ctx->d_ctrl->seam, d_bits_all, rank, world, ctx->stream));
    ctx->launches += 1;
    return phase3_launch(ctx, flags);
}

// One-collective schedule: phase1x -> all-gather of d_record -> phase2x (everything else, no further exchange).
int b2j_strip_phase1x(b2j_ctx *ctx, const uint8_t *d_bgr, size_t step, int width, int rows) {
    if (!ctx || !d_bgr) return B2J_EINVAL;
    REFUSE_GRAY(ctx, "b2j_strip_phase1x");
    CK(cudaSetDevice(ctx->device));
    int rc = enc_alloc(ctx); if (rc) return rc;
    rc = set_strip_geom(ctx, width, rows); if (rc) return rc;
    rc = enc_reset(ctx); if (rc) return rc;
    tick(ctx, 1);
    // symbol counts are always taken: they also give every strip's bit count once the tables are known
    CK(launch_fdct(d_bgr, step, ctx->g, ctx->d_quant, ctx->d_pool, &ctx->d_ctrl->pool_count, ctx->d_recs, ctx->d_ctrl->hist, 1, 0, ctx->g.mcuy, (ctx->debug & 1) ? ctx->d_coef : nullptr, ctx->stream));
    tick(ctx, 2);
    CK(launch_dc_edge_hist(ctx->d_recs, ctx->g, ctx->d_pred_in, ctx->d_ctrl->hist, ctx->d_ctrl->rec.last_dc, 1, ctx->d_pool, 1, &ctx->d_ctrl->rec, 0, ctx->stream));
    ctx->launches += 2;
    if (ctx->peer_world > 0) {   // connected: the record goes straight into every rank's arena
        ctx->xseq++;
        CK(launch_strip_push(&ctx->d_ctrl->rec, ctx->d_peers, ctx->peer_rank, ctx->peer_world, ctx->xseq, ctx->stream));
        ctx->launches += 1;
    }
    tick(ctx, 3);
    return B2J_OK;
}

int b2j_strip_phase2x(b2j_ctx *ctx, const void *d_records_all, int rank, int world, int full_w, int full_h, int flags) {
    if (!ctx || !ctx->enc_ready || rank < 0 || rank >= world || world > 256) return B2J_EINVAL;
    REFUSE_GRAY(ctx, "b2j_strip_phase2x");
    CK(cudaSetDevice(ctx->device));
    const StripRecord *rec = static_cast<const StripRecord *>(d_records_all);
    const uint32_t *xflags = nullptr;
    if (!rec) {   // peer exchange: the records of this image are (or will be) in this rank's arena
        if (ctx->peer_world != world || ctx->peer_rank != rank || ctx->xseq == 0) return B2J_EINVAL;
        const int set = (int)(ctx->xseq % XCHG_SETS);
        rec = ctx->d_arena->rec[set];
        xflags = ctx->d_arena->flags[set];
    }
    CK(launch_strip_merge(rec, rank, world, ctx->d_ctrl->hist, ctx->d_pool, ctx->d_recs, xflags, ctx->xseq, ctx->peer_timeout_ns, &ctx->d_ctrl->err, ctx->stream));
    ctx->launches += 1;
    int rc = strip_phase2(ctx, full_w, full_h); if (rc) return rc;
    CK(launch_strip_seam(rec, rank, world, ctx->d_huff, !(flags & 1), ctx->d_ctrl->seam, ctx->d_ctrl->strip_bits, &ctx->d_ctrl->err, ctx->stream));
    ctx->launches += 1;
    return phase3_launch(ctx, flags, true);
}

// ---- peer-memory exchange set-up (GPUs of one node, one process per GPU) ----------------------------------------
int b2j_peer_export(b2j_ctx *ctx, void *ipc_handle_64, void **d_arena) {
    if (!ctx) return B2J_EINVAL;
    REFUSE_GRAY(ctx, "b2j_peer_export");
    CK(cudaSetDevice(ctx->device));
    if (!ctx->d_arena) {
        CK(cudaMalloc(&ctx->d_arena, sizeof(XchgArena)));
        CK(cudaMemset(ctx->d_arena, 0, sizeof(XchgArena)));
    }
    if (ipc_handle_64) {
        static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size is part of the ABI");
        cudaIpcMemHandle_t h;
        CK(cudaIpcGetMemHandle(&h, ctx->d_arena));
        memcpy(ipc_handle_64, &h, 64);
    }
    if (d_arena) *d_arena = ctx->d_arena;
    return B2J_OK;
}

int b2j_peer_open(b2j_ctx *ctx, const void *ipc_handle_64, void **d_ptr) {
    if (!ctx || !ipc_handle_64 || !d_ptr || ctx->n_opened >= XCHG_MAX_WORLD) return B2J_EINVAL;
    REFUSE_GRAY(ctx, "b2j_peer_open");
    CK(cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    memcpy(&h, ipc_handle_64, 64);
    void *p = nullptr;
    CK(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    ctx->peer_opened[ctx->n_opened++] = p;
    *d_ptr = p;
    return B2J_OK;
}

int b2j_peer_connect(b2j_ctx *ctx, int rank, int world, void *const *d_arenas) {
    if (!ctx || !d_arenas || world < 1 || world > XCHG_MAX_WORLD || rank < 0 || rank >= world || !ctx->d_arena) return B2J_EINVAL;
    REFUSE_GRAY(ctx, "b2j_peer_connect");
    CK(cudaSetDevice(ctx->device));
    XchgArena *host[XCHG_MAX_WORLD];
    for (int r = 0; r < world; r++) {
        host[r] = r == rank ? ctx->d_arena : static_cast<XchgArena *>(d_arenas[r]);
        if (!host[r]) return B2J_EINVAL;
    }
    if (!ctx->d_peers) CK(cudaMalloc(&ctx->d_peers, sizeof(XchgArena *) * XCHG_MAX_WORLD));
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaMemcpy(ctx->d_peers, host, sizeof(XchgArena *) * world, cudaMemcpyHostToDevice));
    CK(cudaMemset(ctx->d_arena, 0, sizeof(XchgArena)));   // every rank connects before any rank encodes (host barrier)
    ctx->peer_rank = rank; ctx->peer_world = world; ctx->xseq = 0;
    const char *e = getenv("B2J_PEER_TIMEOUT_MS");
    ctx->peer_timeout_ns = 1000000ull * (unsigned long long)std::max(1, e ? atoi(e) : 10000);
    return B2J_OK;
}

int b2j_strip_state_get(b2j_ctx *ctx, b2j_strip_state *st) {
    if (!ctx || !st) return B2J_EINVAL;
    REFUSE_GRAY(ctx, "b2j_strip_state_get");
    CK(cudaSetDevice(ctx->device));
    int rc = enc_alloc(ctx); if (rc) return rc;
    st->d_hist = ctx->d_ctrl->hist; st->d_last_dc = ctx->d_ctrl->rec.last_dc; st->d_pred_in = ctx->d_pred_in;
    st->d_strip_bits = ctx->d_ctrl->strip_bits; st->d_out_len = &ctx->d_ctrl->out_len; st->d_out = ctx->d_out;
    st->d_record = &ctx->d_ctrl->rec;
    return B2J_OK;
}

// ------------------------------------------------------------------------------------------ whole-image encode
// Entropy coding of a whole image: k_pack -> k_scan_tiles -> k_stuff (the strips' kernels).
static int enc_tail(b2j_ctx *ctx, int width, int height) {
    int rc = strip_phase1b(ctx); if (rc) return rc;
    rc = strip_phase2(ctx, width, height); if (rc) return rc;
    return strip_phase3(ctx, 0, 0xFF, 3);
}

int b2j_encode_device(b2j_ctx *ctx, const uint8_t *d_bgr, size_t step, int width, int height, const uint8_t **d_out,
                      const uint64_t **d_len) {
    if (!ctx || !d_bgr || step < (size_t)width * chans(ctx)) return B2J_EINVAL;
    CK(cudaSetDevice(ctx->device));
    int rc = enc_alloc(ctx); if (rc) return rc;
    rc = set_strip_geom(ctx, width, height); if (rc) return rc;
    tick(ctx, 0);
    rc = enc_reset(ctx); if (rc) return rc;
    tick(ctx, 1);
    CK(launch_fdct(d_bgr, step, ctx->g, ctx->d_quant, ctx->d_pool, &ctx->d_ctrl->pool_count, ctx->d_recs, ctx->d_ctrl->hist, ctx->p.optimize, 0, ctx->g.mcuy, (ctx->debug & 1) ? ctx->d_coef : nullptr, ctx->stream));
    ctx->launches += 1;
    tick(ctx, 2);
    rc = enc_tail(ctx, width, height); if (rc) return rc;
    if (d_out) *d_out = ctx->d_out;
    if (d_len) *d_len = &ctx->d_ctrl->out_len;
    return B2J_OK;
}

static int fetch_ret(b2j_ctx *ctx) {
    static_assert(sizeof(HostRet) == 40, "HostRet mirrors the fetched block of Ctrl");
    CK(cudaMemcpyAsync(ctx->h_ret, &ctx->d_ctrl->out_len, sizeof(HostRet), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (ctx->h_ret->err || ctx->h_ret->huff_err) {
        snprintf(ctx->err, sizeof(ctx->err), "device check failed: stuff err=%u tables err=%u", ctx->h_ret->err, ctx->h_ret->huff_err);
        return ctx->h_ret->err == 3 ? B2J_ECAPACITY : B2J_EINTERNAL;
    }
    return B2J_OK;
}

static void collect_timings(b2j_ctx *ctx) {
    if (!ctx->timing) return;
    float *dst[7] = {&ctx->tm.h2d, &ctx->tm.fdct, &ctx->tm.hist_edge, &ctx->tm.tables, &ctx->tm.pack, &ctx->tm.scan, &ctx->tm.stuff};
    for (int i = 0; i < 7; i++) { float ms = 0; if (cudaEventElapsedTime(&ms, ctx->ev[i], ctx->ev[i + 1]) != cudaSuccess) { ms = -1; cudaGetLastError(); } *dst[i] = ms; }
    float ms = 0;
    if (cudaEventElapsedTime(&ms, ctx->ev[1], ctx->ev[7]) != cudaSuccess) { ms = -1; cudaGetLastError(); }
    ctx->tm.total = ms;
}

int b2j_encode_finish(b2j_ctx *ctx, size_t *len) {
    if (!ctx) return B2J_EINVAL;
    int rc = fetch_ret(ctx); if (rc) return rc;
    collect_timings(ctx);
    if (len) *len = (size_t)ctx->h_ret->out_len;
    return B2J_OK;
}

static int ensure_img(b2j_ctx *ctx, size_t bytes) {
    if (ctx->d_img_bytes >= bytes) return B2J_OK;
    cudaFree(ctx->d_img); ctx->d_img = nullptr; ctx->d_img_bytes = 0;
    CK(cudaMalloc(&ctx->d_img, bytes));
    ctx->d_img_bytes = bytes;
    return B2J_OK;
}


// ------------------------------------------------------------------------------------------ pageable host buffers
static int ensure_hostpipe(b2j_ctx *ctx, size_t ring_bytes) {
    if (!ctx->pool) {
        unsigned hc = std::thread::hardware_concurrency();
        unsigned want = std::min(12u, std::max(1u, (hc ? hc : 1u) * 3u / 4u));   // 12 of 16 cores measured best on the B200 host
        if (const char *e = getenv("B2J_COPY_THREADS")) want = (unsigned)std::max(1, std::min(64, atoi(e)));
        ctx->pool = new (std::nothrow) CopyPool((int)std::max(1u, want));
        if (!ctx->pool) return B2J_ENOMEM;
    }
    CK(ctx->ring.ensure(ring_bytes));
    return B2J_OK;
}

static constexpr size_t RING_CHUNK = 32u << 20;   // staging granularity of the generic helpers

// rows from the caller's (possibly pageable) memory to the device, asynchronously on `s`
static int upload_2d(b2j_ctx *ctx, uint8_t *d_dst, size_t dstep, const uint8_t *src, size_t sstep, size_t row_bytes, size_t rows,
                     cudaStream_t s) {
    if (!is_pageable_host(src)) {
        CK(cudaMemcpy2DAsync(d_dst, dstep, src, sstep, row_bytes, rows, cudaMemcpyHostToDevice, s));
        return B2J_OK;
    }
    int rc = ensure_hostpipe(ctx, std::max(RING_CHUNK, row_bytes)); if (rc) return rc;
    StageRing &r = ctx->ring;
    const size_t rows_per = std::max<size_t>(1, r.bytes / row_bytes);
    int k = 0;
    for (size_t y = 0; y < rows; y += rows_per, k++) {
        const size_t nr = std::min(rows_per, rows - y);
        const int slot = k % StageRing::N;
        if (r.busy[slot]) CK(cudaEventSynchronize(r.ev[slot]));
        ctx->pool->copy2d(r.buf[slot], row_bytes, src + y * sstep, sstep, row_bytes, nr);
        CK(cudaMemcpy2DAsync(d_dst + y * dstep, dstep, r.buf[slot], row_bytes, row_bytes, nr, cudaMemcpyHostToDevice, s));
        CK(cudaEventRecord(r.ev[slot], s));
        r.busy[slot] = true;
    }
    return B2J_OK;
}

// rows from the device to the caller's (possibly pageable) memory; returns after the data has landed
static int download_2d(b2j_ctx *ctx, uint8_t *dst, size_t hstep, const uint8_t *d_src, size_t dstep, size_t row_bytes, size_t rows,
                       cudaStream_t s) {
    if (!is_pageable_host(dst)) {
        CK(cudaMemcpy2DAsync(dst, hstep, d_src, dstep, row_bytes, rows, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        return B2J_OK;
    }
    int rc = ensure_hostpipe(ctx, std::max(RING_CHUNK, row_bytes)); if (rc) return rc;
    StageRing &r = ctx->ring;
    for (int i = 0; i < StageRing::N; i++) if (r.busy[i]) { CK(cudaEventSynchronize(r.ev[i])); r.busy[i] = false; }
    const size_t rows_per = std::max<size_t>(1, r.bytes / row_bytes);
    const size_t ngroups = (rows + rows_per - 1) / rows_per;
    // group k travels while group k - 1 is copied into the caller's pages
    for (size_t k = 0; k <= ngroups; k++) {
        if (k < ngroups) {
            const size_t y = k * rows_per, nr = std::min(rows_per, rows - y);
            const int slot = (int)(k % StageRing::N);
            CK(cudaMemcpy2DAsync(r.buf[slot], row_bytes, d_src + y * dstep, dstep, row_bytes, nr, cudaMemcpyDeviceToHost, s));
            CK(cudaEventRecord(r.ev[slot], s));
        }
        if (k > 0) {
            const size_t y = (k - 1) * rows_per, nr = std::min(rows_per, rows - y);
            const int slot = (int)((k - 1) % StageRing::N);
            CK(cudaEventSynchronize(r.ev[slot]));
            ctx->pool->copy2d(dst + y * hstep, hstep, r.buf[slot], row_bytes, row_bytes, nr);
        }
    }
    return B2J_OK;
}

// linear buffers go through the same helpers as rows of 1 MB
static int download_linear(b2j_ctx *ctx, uint8_t *dst, const uint8_t *d_src, size_t n, cudaStream_t s) {
    constexpr size_t CH = 1u << 20;
    const size_t rows = n / CH, rem = n - rows * CH;
    int rc = B2J_OK;
    if (rows) rc = download_2d(ctx, dst, CH, d_src, CH, CH, rows, s);
    if (!rc && rem) rc = download_2d(ctx, dst + rows * CH, rem, d_src + rows * CH, rem, rem, 1, s);
    return rc;
}
static int upload_linear(void *user, uint8_t *d_dst, const uint8_t *src, size_t n, cudaStream_t s) {
    b2j_ctx *ctx = static_cast<b2j_ctx *>(user);
    constexpr size_t CH = 1u << 20;
    const size_t rows = n / CH, rem = n - rows * CH;
    int rc = B2J_OK;
    if (rows) rc = upload_2d(ctx, d_dst, CH, src, CH, CH, rows, s);
    if (!rc && rem) rc = upload_2d(ctx, d_dst + rows * CH, rem, src + rows * CH, rem, rem, 1, s);
    return rc;
}

// Rows of a host image (pinned or pageable) -> ctx->d_img in MCU-row groups on the copy stream; the fdct of a group
// starts as soon as its rows have landed. One call issues group `gi` (of `ngroups`): callers that drive several
// contexts interleave the groups of their strips so that every GPU's link is busy. Geometry must be set (ctx->g).
static int upload_fdct_group(b2j_ctx *ctx, const uint8_t *bgr, size_t step, size_t dstep, int gi, int ngroups, int do_hist, bool pageable_in) {
    const Geom &g = ctx->g;
    const int rows_per = (g.mcuy + ngroups - 1) / ngroups;
    const int my0 = gi * rows_per;
    if (my0 >= g.mcuy) return B2J_OK;
    const int mcu_h = 8 * g.vs, width = g.W, height = g.H;
    const size_t row_bytes = (size_t)width * chans(ctx);
    const int nr = std::min(rows_per, g.mcuy - my0);
    const int y0 = my0 * mcu_h, y1 = std::min(height, (my0 + nr) * mcu_h);
    if (gi == 0) {
        CK(cudaEventRecord(ctx->ev_copy[63], ctx->stream));
        CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_copy[63], 0));
    }
    if (pageable_in) {   // copy threads -> pinned ring -> DMA: the group goes up while the next one is being staged
        StageRing &r = ctx->ring;
        const int slot = gi % StageRing::N;
        if (r.busy[slot]) CK(cudaEventSynchronize(r.ev[slot]));
        ctx->pool->copy2d(r.buf[slot], row_bytes, bgr + (size_t)y0 * step, step, row_bytes, y1 - y0);
        CK(cudaMemcpy2DAsync(ctx->d_img + (size_t)y0 * dstep, dstep, r.buf[slot], row_bytes, row_bytes, y1 - y0,
                             cudaMemcpyHostToDevice, ctx->copy_stream));
        CK(cudaEventRecord(r.ev[slot], ctx->copy_stream));
        r.busy[slot] = true;
    } else {
        CK(cudaMemcpy2DAsync(ctx->d_img + (size_t)y0 * dstep, dstep, bgr + (size_t)y0 * step, step, row_bytes, y1 - y0,
                             cudaMemcpyHostToDevice, ctx->copy_stream));
    }
    CK(cudaEventRecord(ctx->ev_copy[gi], ctx->copy_stream));
    CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_copy[gi], 0));
    CK(launch_fdct(ctx->d_img, dstep, g, ctx->d_quant, ctx->d_pool, &ctx->d_ctrl->pool_count, ctx->d_recs, ctx->d_ctrl->hist, do_hist, my0, nr, (ctx->debug & 1) ? ctx->d_coef : nullptr, ctx->stream));
    ctx->launches += 1;
    return B2J_OK;
}

static int upload_groups_of(const Geom &g) { return std::max(1, std::min(32, g.mcuy / 64)); }

// host pixels -> complete JPEG in the context's device buffer; *len = its size (waits for the encode)
int b2j_encode_begin(b2j_ctx *ctx, const uint8_t *bgr, size_t step, int width, int height, size_t *len) {
    if (!ctx || !bgr || !len || step < (size_t)width * chans(ctx)) return B2J_EINVAL;
    CK(cudaSetDevice(ctx->device));
    int rc = enc_alloc(ctx); if (rc) return rc;
    rc = set_strip_geom(ctx, width, height); if (rc) return rc;
    const Geom &g = ctx->g;
    const size_t row_bytes = (size_t)width * chans(ctx);
    const size_t dstep = (row_bytes + 15) & ~(size_t)15;  // 16-byte pitch keeps the TMA path for any width
    rc = ensure_img(ctx, dstep * height); if (rc) return rc;
    tick(ctx, 0);
    rc = enc_reset(ctx); if (rc) return rc;
    // upload in MCU-row groups on the copy stream; the fdct of a group starts as soon as its rows have landed
    const int ngroups = upload_groups_of(g);
    const bool pageable_in = is_pageable_host(bgr);
    if (pageable_in) { rc = ensure_hostpipe(ctx, (size_t)((g.mcuy + ngroups - 1) / ngroups) * 8 * g.vs * row_bytes); if (rc) return rc; }
    tick(ctx, 1);
    for (int gi = 0; gi < ngroups; gi++) { rc = upload_fdct_group(ctx, bgr, step, dstep, gi, ngroups, ctx->p.optimize, pageable_in); if (rc) return rc; }
    tick(ctx, 2);
    rc = enc_tail(ctx, width, height); if (rc) return rc;
    rc = fetch_ret(ctx); if (rc) return rc;
    collect_timings(ctx);
    for (int i = 0; i < StageRing::N; i++) ctx->ring.busy[i] = false;   // every upload has completed (fetch_ret synchronised)
    *len = (size_t)ctx->h_ret->out_len;
    return B2J_OK;
}

// the JPEG of the last b2j_encode_begin -> host memory (pinned or pageable)
int b2j_encode_fetch(b2j_ctx *ctx, uint8_t *out, size_t cap) {
    if (!ctx || !out || !ctx->enc_ready) return B2J_EINVAL;
    CK(cudaSetDevice(ctx->device));
    const size_t n = (size_t)ctx->h_ret->out_len;
    if (n > cap) { snprintf(ctx->err, sizeof(ctx->err), "output needs %zu bytes, buffer has %zu", n, cap); return B2J_ECAPACITY; }
    return download_linear(ctx, out, ctx->d_out, n, ctx->stream);
}

int b2j_encode(b2j_ctx *ctx, const uint8_t *bgr, size_t step, int width, int height, uint8_t *out, size_t cap, size_t *len) {
    if (!out || !len) return B2J_EINVAL;
    size_t n = 0;
    int rc = b2j_encode_begin(ctx, bgr, step, width, height, &n); if (rc) return rc;
    rc = b2j_encode_fetch(ctx, out, cap); if (rc) return rc;
    *len = n;
    return B2J_OK;
}

// ------------------------------------------------------------------------------------------ several GPUs, one process
// One image over the GPUs of one node from a single host thread: MCU-row strips, one context per GPU, the strips'
// records exchanged through peer memory (b2j_peer_*), every strip's rows uploaded in groups over its own GPU's link
// with the fdct of a group behind it, every strip's bytes downloaded straight to their place in the caller's buffer.
struct b2j_multi {
    int n;
    int last_n;                       // strips of the last encode
    size_t off[XCHG_MAX_WORLD + 1];   // byte offsets of the strips' bytes in the stitched stream
    bool shared_device;   // two contexts on one GPU (tests): the host then separates the pushes from the waits
    b2j_ctx *ctx[XCHG_MAX_WORLD];
    char err[256];
};

void b2j_multi_destroy(b2j_multi *m) {
    if (!m) return;
    for (int k = 0; k < m->n; k++) {
        if (m->ctx[k] && k > 0) m->ctx[k]->pool = nullptr;   // the copy threads belong to context 0
        b2j_destroy(m->ctx[k]);
    }
    delete m;
}

const char *b2j_multi_last_error(const b2j_multi *m) { return m ? m->err : "null"; }

int b2j_multi_create(const b2j_params *p, int ngpus, const int *device_ids, b2j_multi **out) {
    if (!p || !out || ngpus < 1 || ngpus > XCHG_MAX_WORLD) return B2J_EINVAL;
    if (p->css == B2J_CSS_GRAY) {   // the strips' records and seams assume three components
        fprintf(stderr, "[b2jpeg] b2j_multi_create: not supported for gray (B2J_CSS_GRAY) images\n");
        return B2J_EINVAL;
    }
    b2j_multi *m = new (std::nothrow) b2j_multi();
    if (!m) return B2J_ENOMEM;
    memset(m, 0, sizeof(*m));
    m->n = ngpus;
    void *arenas[XCHG_MAX_WORLD] = {};
    int rc = B2J_OK;
    for (int k = 0; k < ngpus && !rc; k++) {
        b2j_params pk = *p;
        pk.device = device_ids ? device_ids[k] : k;
        pk.flags |= B2J_FLAG_ENCODE;
        rc = b2j_create(&pk, &m->ctx[k]);
        if (!rc) rc = b2j_peer_export(m->ctx[k], nullptr, &arenas[k]);
    }
    for (int k = 0; k < ngpus && !rc; k++) {   // every GPU stores into every other GPU's arena
        cudaSetDevice(m->ctx[k]->device);
        for (int j = 0; j < ngpus; j++) {
            if (j == k) continue;
            if (m->ctx[j]->device == m->ctx[k]->device) continue;
            const cudaError_t e = cudaDeviceEnablePeerAccess(m->ctx[j]->device, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { snprintf(m->err, sizeof(m->err), "no peer access %d -> %d: %s", m->ctx[k]->device, m->ctx[j]->device, cudaGetErrorString(e)); rc = B2J_ECUDA; break; }
            cudaGetLastError();
        }
    }
    for (int k = 0; k < ngpus && !rc; k++) rc = b2j_peer_connect(m->ctx[k], k, ngpus, arenas);
    for (int k = 0; k < ngpus && !rc; k++)
        for (int j = 0; j < k; j++) if (m->ctx[j]->device == m->ctx[k]->device) m->shared_device = true;
    if (rc) {
        if (!m->err[0]) snprintf(m->err, sizeof(m->err), "context set-up failed (rc=%d)", rc);
        for (int k = 0; k < ngpus; k++) if (m->ctx[k] && m->ctx[k]->err[0]) fprintf(stderr, "[b2jpeg] b2j_multi_create: context %d: %s\n", k, m->ctx[k]->err);
        fprintf(stderr, "[b2jpeg] b2j_multi_create: %s\n", m->err);
        b2j_multi_destroy(m);
        return rc;
    }
    *out = m;
    return B2J_OK;
}

// upload + encode on every GPU; *len = size of the stitched stream (the strips' bytes stay in HBM until b2j_multi_encode_fetch)
int b2j_multi_encode_begin(b2j_multi *m, const uint8_t *bgr, size_t step, int width, int height, size_t *len) {
    if (!m || !bgr || !len || step < (size_t)width * 3) return B2J_EINVAL;
    Geom gw;
    int rc = make_geom(width, height, m->ctx[0]->p.css, &gw); if (rc) return rc;
    const int n = std::min(m->n, gw.mcuy);
    if (n <= 1 || n != m->n) {   // one strip (or fewer MCU rows than GPUs): the single-context path
        rc = b2j_encode_begin(m->ctx[0], bgr, step, width, height, len);
        if (rc) snprintf(m->err, sizeof(m->err), "%s", m->ctx[0]->err);
        m->last_n = 1; m->off[0] = 0; m->off[1] = rc ? 0 : *len;
        return rc;
    }
#define MCK(k, call) do { rc = (call); if (rc) { snprintf(m->err, sizeof(m->err), "gpu %d: %s", (k), m->ctx[k]->err); return rc; } } while (0)
    const int mcu_h = 8 * gw.vs;
    int y0[XCHG_MAX_WORLD + 1];
    for (int k = 0, my = 0; k <= n; k++) { y0[k] = std::min(height, my * mcu_h); my += gw.mcuy / n + (k < gw.mcuy % n ? 1 : 0); }
    const size_t dstep = ((size_t)width * 3 + 15) & ~(size_t)15;
    const bool pageable_in = is_pageable_host(bgr);
    int ngroups = 1;
    for (int k = 0; k < n; k++) {
        b2j_ctx *ctx = m->ctx[k];
        cudaSetDevice(ctx->device);
        MCK(k, enc_alloc(ctx));
        MCK(k, set_strip_geom(ctx, width, y0[k + 1] - y0[k]));
        MCK(k, ensure_img(ctx, dstep * (size_t)(y0[k + 1] - y0[k])));
        MCK(k, enc_reset(ctx));
        ngroups = std::max(ngroups, std::max(1, std::min(16, ctx->g.mcuy / 32)));
    }
    if (pageable_in) {   // one set of copy threads feeds every GPU's staging ring
        for (int k = 0; k < n; k++) {
            b2j_ctx *ctx = m->ctx[k];
            cudaSetDevice(ctx->device);
            if (k > 0 && !ctx->pool) ctx->pool = m->ctx[0]->pool;
            MCK(k, ensure_hostpipe(ctx, (size_t)((ctx->g.mcuy + ngroups - 1) / ngroups) * mcu_h * (size_t)width * 3));
            if (k == 0) for (int j = 1; j < n; j++) if (!m->ctx[j]->pool) m->ctx[j]->pool = ctx->pool;
        }
    }
    // 1. uploads and fdct, group by group across the GPUs (symbol counts are always taken: the strips' bit phases come from them)
    for (int gi = 0; gi < ngroups; gi++)
        for (int k = 0; k < n; k++) {
            cudaSetDevice(m->ctx[k]->device);
            MCK(k, upload_fdct_group(m->ctx[k], bgr + (size_t)y0[k] * step, step, dstep, gi, ngroups, 1, pageable_in));
        }
    // 2. the strips' records into every GPU's arena
    for (int k = 0; k < n; k++) {
        b2j_ctx *ctx = m->ctx[k];
        cudaSetDevice(ctx->device);
        rc = launch_dc_edge_hist(ctx->d_recs, ctx->g, ctx->d_pred_in, ctx->d_ctrl->hist, ctx->d_ctrl->rec.last_dc, 1, ctx->d_pool, 1, &ctx->d_ctrl->rec, 0, ctx->stream) == cudaSuccess ? B2J_OK : B2J_ECUDA;
        if (!rc) { ctx->xseq++; rc = launch_strip_push(&ctx->d_ctrl->rec, ctx->d_peers, ctx->peer_rank, ctx->peer_world, ctx->xseq, ctx->stream) == cudaSuccess ? B2J_OK : B2J_ECUDA; }
        ctx->launches += 2;
        if (rc) { snprintf(m->err, sizeof(m->err), "gpu %d: launch failed", k); return rc; }
    }
    if (m->shared_device)   // kernels that wait on one another must not share a GPU: every record is in place first
        for (int k = 0; k < n; k++) { cudaSetDevice(m->ctx[k]->device); cudaStreamSynchronize(m->ctx[k]->stream); }
    // 3. tables, entropy coding, seam, byte stuffing of every strip (each waits on the device for the others' records)
    for (int k = 0; k < n; k++) {
        cudaSetDevice(m->ctx[k]->device);
        MCK(k, b2j_strip_phase2x(m->ctx[k], nullptr, k, n, width, height, (k == 0 ? 1 : 0) | (k == n - 1 ? 2 : 0)));
    }
    // 4. lengths
    size_t *off = m->off;
    off[0] = 0;
    for (int k = 0; k < n; k++) {
        cudaSetDevice(m->ctx[k]->device);
        MCK(k, fetch_ret(m->ctx[k]));
        for (int i = 0; i < StageRing::N; i++) m->ctx[k]->ring.busy[i] = false;
        off[k + 1] = off[k] + (size_t)m->ctx[k]->h_ret->out_len;
    }
    m->last_n = n;
    *len = off[n];
    return B2J_OK;
#undef MCK
}

// every strip's bytes straight to their place in `out`
int b2j_multi_encode_fetch(b2j_multi *m, uint8_t *out, size_t cap) {
    if (!m || !out || m->last_n < 1) return B2J_EINVAL;
    int rc = B2J_OK;
    const int n = m->last_n;
    const size_t *off = m->off;
#define MCK(k, call) do { rc = (call); if (rc) { snprintf(m->err, sizeof(m->err), "gpu %d: %s", (k), m->ctx[k]->err); return rc; } } while (0)
    if (off[n] > cap) { snprintf(m->err, sizeof(m->err), "output needs %zu bytes, buffer has %zu", off[n], cap); return B2J_ECAPACITY; }
    if (n == 1) {
        rc = b2j_encode_fetch(m->ctx[0], out, cap);
        if (rc) snprintf(m->err, sizeof(m->err), "%s", m->ctx[0]->err);
        return rc;
    }
    const bool pageable_out = is_pageable_host(out);
    for (int k = 0; k < n; k++) {
        b2j_ctx *ctx = m->ctx[k];
        cudaSetDevice(ctx->device);
        if (pageable_out) MCK(k, download_linear(ctx, out + off[k], ctx->d_out, off[k + 1] - off[k], ctx->stream));
        else if (cudaMemcpyAsync(out + off[k], ctx->d_out, off[k + 1] - off[k], cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess) { snprintf(m->err, sizeof(m->err), "gpu %d: download failed", k); return B2J_ECUDA; }
    }
    if (!pageable_out)
        for (int k = 0; k < n; k++) {
            cudaSetDevice(m->ctx[k]->device);
            if (cudaStreamSynchronize(m->ctx[k]->stream) != cudaSuccess) { snprintf(m->err, sizeof(m->err), "gpu %d: %s", k, cudaGetErrorString(cudaGetLastError())); return B2J_ECUDA; }
        }
#undef MCK
    return B2J_OK;
}

int b2j_multi_encode(b2j_multi *m, const uint8_t *bgr, size_t step, int width, int height, uint8_t *out, size_t cap, size_t *len) {
    if (!out || !len) return B2J_EINVAL;
    size_t n = 0;
    int rc = b2j_multi_encode_begin(m, bgr, step, width, height, &n); if (rc) return rc;
    rc = b2j_multi_encode_fetch(m, out, cap); if (rc) return rc;
    *len = n;
    return B2J_OK;
}

int b2j_last_timings(b2j_ctx *ctx, b2j_timings *t) { if (!ctx || !t) return B2J_EINVAL; *t = ctx->tm; return B2J_OK; }

// ------------------------------------------------------------------------------------------ decode
static int dec_ensure(b2j_ctx *ctx) {
    if (ctx->dec) return B2J_OK;
    // a gray context also decodes the Y plane of colour files of its configured size: room for their blocks (4:4:4 has
    // the most per pixel)
    int nb = ctx->cap_g.nblocks;
    Geom g444;
    if (ctx->p.css == B2J_CSS_GRAY && make_geom(ctx->cap_g.W, ctx->cap_g.H, B2J_CSS_444, &g444) == B2J_OK) nb = g444.nblocks;
    ctx->dec = dec_create(nb, ctx->err, sizeof(ctx->err));
    if (ctx->dec) dec_set_uploader(ctx->dec, upload_linear, ctx);   // pageable JPEG bytes go up through the staging ring
    return ctx->dec ? B2J_OK : B2J_ECUDA;
}

int b2j_peek(const uint8_t *jpg, size_t len, int *width, int *height, int *css) {
    JpegInfo info;
    const int rc = parse_jpeg(jpg, len, &info);
    if (rc) return rc;
    if (width) *width = info.W;
    if (height) *height = info.H;
    if (css) *css = info.css;
    return B2J_OK;
}

// A colour context takes three-component files only; a gray context takes one-component files and the Y plane of
// three-component ones (libjpeg's JCS_GRAYSCALE output)
static int check_components(b2j_ctx *ctx, int file_css) {
    if (file_css != B2J_CSS_GRAY || chans(ctx) == 1) return B2J_OK;
    snprintf(ctx->err, sizeof(ctx->err), "one-component (gray) JPEG: decode it on a B2J_CSS_GRAY context");
    return B2J_EFORMAT;
}

// sequential files: asynchronous (careful = false: dec_check may ask for a checked retry); progressive files: scan by
// scan (dec_prog.cu), synchronous
static int decode_parsed(b2j_ctx *ctx, const uint8_t *jpg, size_t len, const JpegInfo &info, uint8_t *d_bgr, size_t step, bool careful,
                         int scale, const uint8_t *d_scan_src = nullptr) {
    if (step < (size_t)dec_scaled_size(info.W, scale) * chans(ctx)) return B2J_EINVAL;
    int rc = dec_ensure(ctx); if (rc) return rc;
    Geom g; rc = make_geom(info.W, info.H, info.css, &g); if (rc) return rc;
    if (info.progressive) return dec_run_progressive(ctx->dec, jpg, len, info, g, d_bgr, step, chans(ctx) == 1, ctx->stream, &ctx->launches, scale);
    dec_set_spec_launches(ctx->dec, (ctx->debug & 4) ? 1 : 3);
    return dec_run(ctx->dec, jpg, len, info, g, d_bgr, step, chans(ctx) == 1, ctx->stream, ctx->timing ? &ctx->tm : nullptr,
                   &ctx->launches, careful, d_scan_src, scale);
}

static int parse_for(b2j_ctx *ctx, const uint8_t *jpg, size_t len, JpegInfo *info, int *width, int *height) {
    int rc = parse_jpeg(jpg, len, info);
    if (rc) { snprintf(ctx->err, sizeof(ctx->err), "unsupported or corrupt JPEG (parse rc=%d)", rc); return B2J_EFORMAT; }
    rc = check_components(ctx, info->css); if (rc) return rc;
    if (info->progressive && info->smoothed[chans(ctx) == 1]) {
        snprintf(ctx->err, sizeof(ctx->err), "incomplete progressive JPEG (low-frequency coefficients unfinished): "
                 "libjpeg would block-smooth it, which this decoder does not do");
        return B2J_EFORMAT;
    }
    if (width) *width = dec_scaled_size(info->W, ctx->dec_scale);
    if (height) *height = dec_scaled_size(info->H, ctx->dec_scale);
    return B2J_OK;
}

// ctx->d_recon of at least `bytes`: b2j_decode's image before it is downloaded, the secondary compression's reconstruction
static int ensure_recon(b2j_ctx *ctx, size_t bytes) {
    if (ctx->d_recon_bytes >= bytes) return B2J_OK;
    cudaFree(ctx->d_recon); ctx->d_recon = nullptr; ctx->d_recon_bytes = 0;
    CK(cudaMalloc(&ctx->d_recon, bytes));
    ctx->d_recon_bytes = bytes;
    return B2J_OK;
}

int b2j_decode_device(b2j_ctx *ctx, const uint8_t *jpg, size_t len, uint8_t *d_bgr, size_t step, int *width, int *height) {
    if (!ctx || !jpg) return B2J_EINVAL;
    CK(cudaSetDevice(ctx->device));
    JpegInfo info;
    int rc = parse_for(ctx, jpg, len, &info, width, height);
    if (rc || !d_bgr) return rc;
    // one decode in flight per context: an unfinished predecessor is finished (validated, retried if needed) first
    if (ctx->last_jpg) { rc = b2j_decode_finish(ctx); if (rc) return rc; }
    // progressive files decode synchronously: nothing is left for b2j_decode_finish
    if (info.progressive) return decode_parsed(ctx, jpg, len, info, d_bgr, step, false, ctx->dec_scale);
    // remembered for b2j_decode_finish: the caller keeps `jpg` alive until then
    ctx->last_jpg = jpg; ctx->last_len = len; ctx->last_bgr = d_bgr; ctx->last_step = step; ctx->last_scale = ctx->dec_scale;
    return decode_parsed(ctx, jpg, len, info, d_bgr, step, false, ctx->last_scale);
}

// A baseline JPEG whose entropy-coded segment is already in DEVICE memory (the output of b2j_encode_device, a slice
// of a stream with restart intervals, ...): `hdr` = the file's bytes from SOI up to and including the SOS header (host
// memory, a few hundred bytes), d_scan = the stuffed scan bytes up to the terminating marker. height_override > 0
// replaces the frame height: whole restart intervals of whole MCU rows decode as an image of their own (multi-GPU
// decode of one image, strips.StripDecoder). Synchronous: validated (and redone with the checked schedule if needed)
// before it returns.
int b2j_decode_scan_device(b2j_ctx *ctx, const uint8_t *hdr, size_t hdr_len, const uint8_t *d_scan, size_t scan_len,
                           int height_override, uint8_t *d_bgr, size_t step, int *width, int *height) {
    if (!ctx || !hdr || !d_scan || !d_bgr || scan_len == 0) return B2J_EINVAL;
    CK(cudaSetDevice(ctx->device));
    if (ctx->last_jpg) { int rf = b2j_decode_finish(ctx); if (rf) return rf; }
    JpegInfo info;
    int rc = parse_for(ctx, hdr, hdr_len, &info, nullptr, nullptr); if (rc) return rc;
    if (info.progressive) { snprintf(ctx->err, sizeof(ctx->err), "progressive JPEG: one scan in device memory cannot be decoded"); return B2J_EFORMAT; }
    JpegScan &sc = info.scans[0];
    if (sc.seg_off != hdr_len) { snprintf(ctx->err, sizeof(ctx->err), "hdr must end with the SOS header"); return B2J_EINVAL; }
    if (height_override > 0) info.H = height_override;
    sc.seg_off = 0; sc.seg_len = scan_len;
    const int scale = ctx->dec_scale;
    if (width) *width = dec_scaled_size(info.W, scale);
    if (height) *height = dec_scaled_size(info.H, scale);
    for (int attempt = 0; attempt < 2; attempt++) {
        rc = decode_parsed(ctx, hdr, hdr_len, info, d_bgr, step, attempt == 1, scale, d_scan); if (rc) return rc;
        rc = dec_check(ctx->dec, ctx->err, sizeof(ctx->err));
        if (rc != DEC_RETRY) break;
    }
    return rc;
}

int b2j_decode_finish(b2j_ctx *ctx) {
    if (!ctx) return B2J_EINVAL;
    if (!ctx->dec || !ctx->last_jpg) return B2J_OK;
    CK(cudaSetDevice(ctx->device));
    int rc = dec_check(ctx->dec, ctx->err, sizeof(ctx->err));
    if (rc == DEC_RETRY) {   // the speculative synchronisation schedule was too short for this stream: decode again, checked
        JpegInfo info;
        rc = parse_for(ctx, ctx->last_jpg, ctx->last_len, &info, nullptr, nullptr); if (rc) return rc;
        rc = decode_parsed(ctx, ctx->last_jpg, ctx->last_len, info, ctx->last_bgr, ctx->last_step, true, ctx->last_scale); if (rc) return rc;
        rc = dec_check(ctx->dec, ctx->err, sizeof(ctx->err));
    }
    ctx->last_jpg = nullptr;
    return rc;
}

int b2j_decode(b2j_ctx *ctx, const uint8_t *jpg, size_t len, uint8_t *bgr, size_t step, int *width, int *height) {
    if (!ctx || !jpg) return B2J_EINVAL;
    CK(cudaSetDevice(ctx->device));
    JpegInfo info;
    int rc = parse_for(ctx, jpg, len, &info, width, height);
    if (rc || !bgr) return rc;
    const int ch = chans(ctx), scale = ctx->dec_scale, ow = dec_scaled_size(info.W, scale), oh = dec_scaled_size(info.H, scale);
    if (step < (size_t)ow * ch) return B2J_EINVAL;
    const size_t dstep = ((size_t)ow * ch + 15) & ~(size_t)15;
    rc = ensure_recon(ctx, dstep * oh); if (rc) return rc;
    for (int attempt = 0; attempt < 2; attempt++) {
        rc = decode_parsed(ctx, jpg, len, info, ctx->d_recon, dstep, attempt == 1, scale);
        if (rc) return rc;
        rc = download_2d(ctx, bgr, step, ctx->d_recon, dstep, (size_t)ow * ch, oh, ctx->stream); if (rc) return rc;
        rc = dec_check(ctx->dec, ctx->err, sizeof(ctx->err));
        if (rc != DEC_RETRY) break;   // else: the speculative synchronisation schedule was too short: once more, checked
    }
    return rc;
}

// ------------------------------------------------------------------------------------------ diff / PSNR / secondary
int b2j_diff_psnr_device(b2j_ctx *ctx, const uint8_t *d_a, const uint8_t *d_b, size_t n, int mode, uint8_t *d_out,
                         const uint64_t **d_ssd) {
    if (!ctx || !d_a || !d_b || (mode != 0 && mode != 1)) return B2J_EINVAL;
    int rc = enc_alloc(ctx); if (rc) return rc;
    CK(cudaMemsetAsync(&ctx->d_ctrl->ssd, 0, 8, ctx->stream));
    CK(launch_diff_psnr(d_a, d_b, n, mode, d_out, &ctx->d_ctrl->ssd, ctx->stream));
    ctx->launches += 1;
    if (d_ssd) *d_ssd = &ctx->d_ctrl->ssd;
    return B2J_OK;
}

static double psnr_from_ssd(uint64_t ssd, size_t n) {
    const double diff = sqrt((double)ssd / (double)n);
    return 20.0 * log10(255.0 / (diff + 2.220446049250313e-16));  // cv::PSNR
}

static int diff_psnr_host(b2j_ctx *ctx, const uint8_t *a, const uint8_t *b, size_t n, int mode, uint8_t *out, double *psnr, uint64_t *ssd) {
    if (!ctx || !a || !b || n == 0) return B2J_EINVAL;
    CK(cudaSetDevice(ctx->device));
    uint8_t *d = nullptr;
    CK(cudaMalloc(&d, 3 * ((n + 15) & ~(size_t)15)));
    const size_t pitch = (n + 15) & ~(size_t)15;
    int rc = B2J_OK;
    do {
        if (cudaMemcpyAsync(d, a, n, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess ||
            cudaMemcpyAsync(d + pitch, b, n, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess) { rc = B2J_ECUDA; break; }
        rc = b2j_diff_psnr_device(ctx, d, d + pitch, n, mode, out ? d + 2 * pitch : nullptr, nullptr);
        if (rc) break;
        if (out && cudaMemcpyAsync(out, d + 2 * pitch, n, cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess) { rc = B2J_ECUDA; break; }
        if (cudaMemcpyAsync(&ctx->h_ret->ssd, &ctx->d_ctrl->ssd, 8, cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess ||
            cudaStreamSynchronize(ctx->stream) != cudaSuccess) { rc = B2J_ECUDA; break; }
        if (ssd) *ssd = ctx->h_ret->ssd;
        if (psnr) *psnr = psnr_from_ssd(ctx->h_ret->ssd, n);
    } while (0);
    cudaFree(d);
    if (rc == B2J_ECUDA) snprintf(ctx->err, sizeof(ctx->err), "%s in diff/psnr", cudaGetErrorString(cudaGetLastError()));
    return rc;
}

int b2j_diff(b2j_ctx *ctx, const uint8_t *a, const uint8_t *b, size_t n, int mode, uint8_t *out) {
    if (!out || (mode != 0 && mode != 1)) return B2J_EINVAL;
    return diff_psnr_host(ctx, a, b, n, mode, out, nullptr, nullptr);
}

int b2j_psnr(b2j_ctx *ctx, const uint8_t *a, const uint8_t *b, size_t n, double *psnr, uint64_t *ssd) {
    return diff_psnr_host(ctx, a, b, n, 0, nullptr, psnr, ssd);
}

// Reconstruction without an entropy decode: the pixels every decoder will produce from the LAST encode of this
// context, from the quantised coefficients k_fdct kept (B2J_DEBUG_COEF set before that encode): de-quantise + islow
// IDCT + fancy upsampling + YCbCr->BGR, the decoder's own kernels. Asynchronous on the context's stream.
static int recon_layout(b2j_ctx *ctx, uint8_t **py, uint8_t **pcb, uint8_t **pcr) {
    const Geom &g = ctx->g;
    const size_t cs = (size_t)g.mcux * 8;   // chroma row pitch; one spare row above and below every chroma plane (halos)
    const size_t ysz = ((size_t)g.mcux * 8 * g.hs * g.mcuy * 8 * g.vs + 63) & ~(size_t)63;
    const size_t csz = (cs * ((size_t)g.mcuy * 8 + 2) + 63) & ~(size_t)63;
    if (ctx->rplanes_bytes < ysz + 2 * csz + 256) {
        cudaFree(ctx->d_rplanes); ctx->d_rplanes = nullptr; ctx->rplanes_bytes = 0;
        CK(cudaMalloc(&ctx->d_rplanes, ysz + 2 * csz + 256));
        ctx->rplanes_bytes = ysz + 2 * csz + 256;
    }
    *py = ctx->d_rplanes; *pcb = *py + ysz + cs; *pcr = *pcb + csz;
    return B2J_OK;
}

// First half of the reconstruction: de-quantise + IDCT of the coefficients the last encode kept -> sample planes.
// A strip of a larger image (several GPUs) then fetches one chroma row from each neighbour strip into its halo rows
// before b2j_reconstruct_color: the vertical chroma filter of 4:2:0 / 4:4:0 looks one row across the border.
int b2j_reconstruct_planes(b2j_ctx *ctx, b2j_recon_planes *out) {
    if (!ctx) return B2J_EINVAL;
    REFUSE_GRAY(ctx, "b2j_reconstruct_planes");
    if (!ctx->enc_ready || !(ctx->debug & 1) || !ctx->d_coef) { snprintf(ctx->err, sizeof(ctx->err), "b2j_reconstruct_* needs an encode with B2J_DEBUG_COEF set"); return B2J_EINVAL; }
    const Geom &g = ctx->g;
    CK(cudaSetDevice(ctx->device));
    uint8_t *py, *pcb, *pcr;
    int rc = recon_layout(ctx, &py, &pcb, &pcr); if (rc) return rc;
    if (!ctx->d_rtb) {
        std::vector<uint8_t> h(dec_tables_size(), 0);
        DecTables *t = reinterpret_cast<DecTables *>(h.data());
        memcpy(t->q, ctx->hq.q, sizeof(t->q));
        CK(cudaMalloc(&ctx->d_rtb, dec_tables_size()));
        CK(cudaMemcpy(ctx->d_rtb, h.data(), h.size(), cudaMemcpyHostToDevice));
    }
    CK(launch_idct(ctx->d_coef, nullptr, g, ctx->d_rtb, py, pcb, pcr, 0, ctx->stream));
    ctx->launches += 1;
    if (out) {
        const size_t cs = (size_t)g.mcux * 8;
        const int dh = g.dh[1];
        out->row_bytes = (size_t)g.dw[1];
        out->cb_first = pcb; out->cr_first = pcr;
        out->cb_last = pcb + (size_t)(dh - 1) * cs; out->cr_last = pcr + (size_t)(dh - 1) * cs;
        out->cb_halo_top = pcb - cs; out->cr_halo_top = pcr - cs;
        out->cb_halo_bottom = pcb + (size_t)dh * cs; out->cr_halo_bottom = pcr + (size_t)dh * cs;
    }
    return B2J_OK;
}

// Second half: upsampling + colour conversion of the planes. halo_top / halo_bottom != 0: the halo rows are filled.
int b2j_reconstruct_color(b2j_ctx *ctx, uint8_t *d_bgr, size_t step, int halo_top, int halo_bottom) {
    if (!ctx || !d_bgr) return B2J_EINVAL;
    REFUSE_GRAY(ctx, "b2j_reconstruct_color");
    if (!ctx->d_rplanes) return B2J_EINVAL;
    const Geom &g = ctx->g;
    if (step < (size_t)g.W * 3) return B2J_EINVAL;
    CK(cudaSetDevice(ctx->device));
    uint8_t *py, *pcb, *pcr;
    int rc = recon_layout(ctx, &py, &pcb, &pcr); if (rc) return rc;
    CK(launch_upcolor(py, pcb, pcr, g, d_bgr, step, ctx->stream, halo_top, halo_bottom));
    ctx->launches += 1;
    return B2J_OK;
}

int b2j_reconstruct_device(b2j_ctx *ctx, uint8_t *d_bgr, size_t step) {
    if (!ctx || !d_bgr) return B2J_EINVAL;
    REFUSE_GRAY(ctx, "b2j_reconstruct_device");
    int rc = b2j_reconstruct_planes(ctx, nullptr); if (rc) return rc;
    return b2j_reconstruct_color(ctx, d_bgr, step, 0, 0);
}

// Secondary compression, device resident and asynchronous: encode -> reconstruct from the encoder's own coefficients
// -> difference map + SSD -> encode(difference). Nothing leaves the device, nothing is entropy-decoded, the host is
// not waited for; b2j_secondary_finish returns the two lengths and the PSNR.
int b2j_secondary_device(b2j_ctx *ctx, const uint8_t *d_bgr, size_t step, int width, int height, int diff_mode,
                         const uint8_t **d_jpg1, const uint8_t **d_jpg2, const uint8_t **d_recon, const uint8_t **d_diff) {
    if (!ctx) return B2J_EINVAL;
    REFUSE_GRAY(ctx, "b2j_secondary_device");
    if (!d_bgr || step != (size_t)width * 3 || (diff_mode != 0 && diff_mode != 1)) return B2J_EINVAL;   // contiguous rows
    CK(cudaSetDevice(ctx->device));
    const size_t bytes = (size_t)width * 3 * height;
    int rc = ensure_recon(ctx, bytes); if (rc) return rc;
    if (ctx->d_diff_bytes < bytes) { cudaFree(ctx->d_diff); ctx->d_diff = nullptr; ctx->d_diff_bytes = 0; CK(cudaMalloc(&ctx->d_diff, bytes)); ctx->d_diff_bytes = bytes; }
    if (!ctx->second) {
        b2j_params p2 = ctx->p; p2.flags = 0; p2.device = ctx->device;
        int rc2 = b2j_create(&p2, &ctx->second); if (rc2) return rc2;
    }
    b2j_set_stream(ctx->second, ctx->stream);
    const int dbg = ctx->debug;
    ctx->debug |= 1;
    rc = ensure_debug(ctx);
    const uint8_t *o1 = nullptr, *o2 = nullptr; const uint64_t *l1, *l2;
    if (!rc) rc = b2j_encode_device(ctx, d_bgr, step, width, height, &o1, &l1);
    if (!rc) rc = b2j_reconstruct_device(ctx, ctx->d_recon, (size_t)width * 3);
    ctx->debug = dbg;
    if (rc) return rc;
    rc = b2j_diff_psnr_device(ctx, d_bgr, ctx->d_recon, bytes, diff_mode, ctx->d_diff, nullptr); if (rc) return rc;
    rc = b2j_encode_device(ctx->second, ctx->d_diff, (size_t)width * 3, width, height, &o2, &l2);
    if (rc) { snprintf(ctx->err, sizeof(ctx->err), "secondary encode: %s", ctx->second->err); return rc; }
    if (d_jpg1) *d_jpg1 = o1;
    if (d_jpg2) *d_jpg2 = o2;
    if (d_recon) *d_recon = ctx->d_recon;
    if (d_diff) *d_diff = ctx->d_diff;
    ctx->sec_pixels = (size_t)width * height * 3;
    return B2J_OK;
}

int b2j_secondary_finish(b2j_ctx *ctx, size_t *len1, size_t *len2, double *psnr, uint64_t *ssd) {
    if (!ctx) return B2J_EINVAL;
    REFUSE_GRAY(ctx, "b2j_secondary_finish");
    if (!ctx->second) return B2J_EINVAL;
    CK(cudaSetDevice(ctx->device));
    // the SSD lives in the first encoder's control block: b2j_diff_psnr_device ran after its encode was queued, and
    // fetch_ret copies the block (length, checks, SSD) in one go
    int rc = fetch_ret(ctx); if (rc) return rc;
    if (len1) *len1 = (size_t)ctx->h_ret->out_len;
    if (ssd) *ssd = ctx->h_ret->ssd;
    if (psnr) *psnr = psnr_from_ssd(ctx->h_ret->ssd, ctx->sec_pixels);
    size_t n2 = 0;
    rc = b2j_encode_finish(ctx->second, &n2);
    if (rc) { snprintf(ctx->err, sizeof(ctx->err), "secondary encode: %s", ctx->second->err); return rc; }
    if (len2) *len2 = n2;
    return B2J_OK;
}

int b2j_secondary(b2j_ctx *ctx, const uint8_t *bgr, size_t step, int width, int height, int diff_mode, uint8_t *jpg1,
                  size_t cap1, size_t *len1, uint8_t *jpg2, size_t cap2, size_t *len2, uint8_t *recon, size_t recon_step,
                  double *psnr) {
    if (!ctx) return B2J_EINVAL;
    REFUSE_GRAY(ctx, "b2j_secondary");
    if (!bgr || step < (size_t)width * 3 || (diff_mode != 0 && diff_mode != 1)) return B2J_EINVAL;
    CK(cudaSetDevice(ctx->device));
    int rc = enc_alloc(ctx); if (rc) return rc;
    // host pixels -> device (contiguous rows), then everything stays there: b2j_secondary_device
    const size_t row = (size_t)width * 3;
    rc = ensure_img(ctx, row * height); if (rc) return rc;
    rc = upload_2d(ctx, ctx->d_img, row, bgr, step, row, height, ctx->stream); if (rc) return rc;
    const uint8_t *dj1 = nullptr, *dj2 = nullptr, *drec = nullptr;
    rc = b2j_secondary_device(ctx, ctx->d_img, row, width, height, diff_mode, &dj1, &dj2, &drec, nullptr); if (rc) return rc;
    size_t n1 = 0, n2 = 0;
    rc = b2j_secondary_finish(ctx, &n1, &n2, psnr, nullptr); if (rc) return rc;
    for (int i = 0; i < StageRing::N; i++) ctx->ring.busy[i] = false;   // every upload has completed
    if (len1) *len1 = n1;
    if (len2) *len2 = n2;
    if (jpg1) { if (n1 > cap1) return B2J_ECAPACITY; rc = download_linear(ctx, jpg1, dj1, n1, ctx->stream); if (rc) return rc; }
    if (jpg2) { if (n2 > cap2) return B2J_ECAPACITY; rc = download_linear(ctx, jpg2, dj2, n2, ctx->stream); if (rc) return rc; }
    if (recon) { rc = download_2d(ctx, recon, recon_step, drec, row, row, height, ctx->stream); if (rc) return rc; }
    return B2J_OK;
}

// the results of the last b2j_secondary / b2j_secondary_device (+ _finish) -> host memory; any pointer may be NULL
int b2j_secondary_fetch(b2j_ctx *ctx, uint8_t *jpg1, size_t cap1, uint8_t *jpg2, size_t cap2, uint8_t *recon, size_t recon_step) {
    if (!ctx) return B2J_EINVAL;
    REFUSE_GRAY(ctx, "b2j_secondary_fetch");
    if (!ctx->second || !ctx->enc_ready) return B2J_EINVAL;
    CK(cudaSetDevice(ctx->device));
    const size_t n1 = (size_t)ctx->h_ret->out_len, n2 = (size_t)ctx->second->h_ret->out_len;
    int rc = B2J_OK;
    if (jpg1) { if (n1 > cap1) return B2J_ECAPACITY; rc = download_linear(ctx, jpg1, ctx->d_out, n1, ctx->stream); if (rc) return rc; }
    if (jpg2) { if (n2 > cap2) return B2J_ECAPACITY; rc = download_linear(ctx, jpg2, ctx->second->d_out, n2, ctx->stream); if (rc) return rc; }
    if (recon) {
        const size_t row = (size_t)ctx->g.W * 3;
        if (recon_step < row) return B2J_EINVAL;
        rc = download_2d(ctx, recon, recon_step, ctx->d_recon, row, row, ctx->g.H, ctx->stream);
    }
    return rc;
}

// ------------------------------------------------------------------------------------------ introspection
int b2j_debug_read(b2j_ctx *ctx, int what, void *dst, size_t cap, size_t *len) {
    if (!ctx || !dst) return B2J_EINVAL;
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    const void *src = nullptr; size_t n = 0;
    switch (what) {
    case B2J_DBG_COEF: if (!ctx->enc_ready || !ctx->d_coef) return B2J_EINVAL; src = ctx->d_coef; n = (size_t)ctx->g.nblocks * 128; break;
    case B2J_DBG_HIST: if (!ctx->enc_ready) return B2J_EINVAL; src = ctx->d_ctrl->hist; n = 4 * 257 * 4; break;
    case B2J_DBG_TABLES: if (!ctx->enc_ready) return B2J_EINVAL; src = ctx->d_huff; n = sizeof(HuffDev); break;
    case B2J_DBG_TILE_BITS: if (!ctx->enc_ready) return B2J_EINVAL; src = ctx->d_tile_bits; n = (size_t)ctx->g.ntiles * 4; break;
    case B2J_DBG_TOKEN_COUNT: if (!ctx->enc_ready) return B2J_EINVAL; src = &ctx->d_ctrl->pool_count; n = 4; break;
    case B2J_DBG_TOKENS: { if (!ctx->enc_ready) return B2J_EINVAL; uint32_t cnt = 0; CK(cudaMemcpy(&cnt, &ctx->d_ctrl->pool_count, 4, cudaMemcpyDeviceToHost)); src = ctx->d_pool; n = (size_t)cnt * 4; break; }
    case B2J_DBG_TILE_RECS: if (!ctx->enc_ready) return B2J_EINVAL; src = ctx->d_recs; n = (size_t)ctx->g.ntiles * sizeof(TileRec); break;
    case B2J_DBG_SLOTS: if (!ctx->enc_ready) return B2J_EINVAL; src = ctx->d_slots; n = (size_t)ctx->g.ntiles * SLOT_WORDS * 4; break;
    case B2J_DBG_DEC_COEF: if (!ctx->dec) return B2J_EINVAL; src = dec_coef_ptr(ctx->dec, &n); break;
    default: return B2J_EINVAL;
    }
    if (len) *len = n;
    if (n > cap) return B2J_ECAPACITY;
    CK(cudaMemcpy(dst, src, n, cudaMemcpyDeviceToHost));
    return B2J_OK;
}

}  // extern "C"
