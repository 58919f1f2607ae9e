// dec.cu -- host side of the decoder: buffers, stage sequencing, the synchronisation loop.
// Mirrors NvjpegCompressRunnerImpl::DecodeWorker (reference ImageCompressorImpl.cu:311-385) with nvJPEG replaced by
// this library's kernels; output planes are never materialised as three B/G/R planes (the reference's
// getCVImageOnCPU :184-232 step disappears into k_upcolor's interleaved store).
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "dec.h"
#include "dec_kernels.h"

namespace b2j {

struct DecCtrl {
    uint64_t u_len;
    uint64_t avail;      // bytes de-stuffed so far (pipelined front end)
    uint32_t ticket[8];  // 0 unused, 1 nblk scan, 2..4 dc scan
    uint32_t dticket[32];  // one counter per de-stuff launch
    uint32_t err;
    uint32_t changed;
    uint32_t changed_alt;   // the launches of the fixed schedule alternate between the two flags
    uint32_t nmark;      // restart markers found by k_destuff
};

struct Decoder {
    int nblocks_cap = 0;
    // entropy segment
    uint8_t *d_scan = nullptr, *d_u = nullptr;
    size_t scan_cap = 0;
    uint64_t *d_desc = nullptr;
    size_t desc_cap = 0;       // entries per descriptor array (5 arrays)
    uint64_t *d_st_in = nullptr, *d_st_out = nullptr;
    uint32_t *d_nblk = nullptr, *d_blk_start = nullptr;
    uint8_t *d_done = nullptr;   // per decoder chunk (256 subsequences): first synchronisation pass has run
    uint32_t *d_bnd = nullptr;   // restart intervals: start offsets in the unstuffed stream (k_destuff<true>)
    size_t bnd_cap = 0;
    size_t nsub_cap = 0;
    cudaStream_t up_stream = nullptr;   // uploads of the scan pieces
    cudaEvent_t ev_up[33] = {};
    DecCtrl *d_ctrl = nullptr;
    void *d_tb = nullptr;
    void *h_tb = nullptr;      // pinned
    uint32_t *h_flag = nullptr;  // pinned: [0] changed, [1] err
    int16_t *d_coef = nullptr;
    int16_t *d_dc = nullptr;     // one DC per block: differences from k_dec_write, un-differenced in place by k_dc_scan
    uint8_t *d_planes = nullptr;
    size_t planes_cap = 0;
    cudaEvent_t ev[8];
    int last_rounds = 0;
    char *err;
    size_t errlen;
    cudaStream_t last_stream = nullptr;
    bool in_flight = false;     // a decode was issued and dec_check has not drained it yet
    dec_upload_fn upload = nullptr;
    void *upload_user = nullptr;
    bool speculated = false;   // the last run issued a fixed number of synchronisation launches without looking
    int spec_launches = 3;     // that number (tests shorten it to force the retry path)
    int long_group = 0;        // B2J_DEC_GROUP: subsequences per thread of k_dec_sync_long (0: chosen per stream)
};

#define DCK(call)                                                                                                  \
    do {                                                                                                           \
        cudaError_t _e = (call);                                                                                   \
        if (_e != cudaSuccess) {                                                                                   \
            snprintf(d->err, d->errlen, "%s at %s:%d", cudaGetErrorString(_e), __FILE__, __LINE__);                 \
            return B2J_ECUDA;                                                                                      \
        }                                                                                                          \
    } while (0)

Decoder *dec_create(int nblocks_cap, char *err, size_t errlen) {
    Decoder *d = new Decoder();
    d->nblocks_cap = nblocks_cap;
    d->err = err;
    d->errlen = errlen;
    if (const char *e = getenv("B2J_DEC_GROUP")) d->long_group = atoi(e);
    bool ok = cudaMalloc(&d->d_ctrl, sizeof(DecCtrl)) == cudaSuccess && cudaMalloc(&d->d_tb, dec_tables_size()) == cudaSuccess &&
              cudaHostAlloc(&d->h_tb, dec_tables_size(), cudaHostAllocDefault) == cudaSuccess &&
              cudaHostAlloc(&d->h_flag, 16, cudaHostAllocDefault) == cudaSuccess &&
              cudaMalloc(&d->d_coef, (size_t)nblocks_cap * 128) == cudaSuccess &&
              cudaMalloc(&d->d_dc, (size_t)nblocks_cap * 2 + 64) == cudaSuccess;
    for (auto &e : d->ev) ok = ok && cudaEventCreate(&e) == cudaSuccess;
    ok = ok && cudaStreamCreateWithFlags(&d->up_stream, cudaStreamNonBlocking) == cudaSuccess;
    for (auto &e : d->ev_up) ok = ok && cudaEventCreateWithFlags(&e, cudaEventDisableTiming) == cudaSuccess;
    if (!ok) {
        snprintf(err, errlen, "decoder allocation failed: %s", cudaGetErrorString(cudaGetLastError()));
        dec_destroy(d);
        return nullptr;
    }
    return d;
}

void dec_destroy(Decoder *d) {
    if (!d) return;
    cudaFree(d->d_scan); cudaFree(d->d_u); cudaFree(d->d_desc); cudaFree(d->d_st_in); cudaFree(d->d_st_out);
    cudaFree(d->d_nblk); cudaFree(d->d_blk_start); cudaFree(d->d_ctrl); cudaFree(d->d_tb); cudaFree(d->d_coef); cudaFree(d->d_dc);
    cudaFree(d->d_planes);
    if (d->h_tb) cudaFreeHost(d->h_tb);
    if (d->h_flag) cudaFreeHost(d->h_flag);
    for (auto &e : d->ev) if (e) cudaEventDestroy(e);
    for (auto &e : d->ev_up) if (e) cudaEventDestroy(e);
    if (d->up_stream) cudaStreamDestroy(d->up_stream);
    cudaFree(d->d_done);
    cudaFree(d->d_bnd);
    delete d;
}

void dec_set_uploader(Decoder *d, dec_upload_fn fn, void *user) { d->upload = fn; d->upload_user = user; }
void dec_set_spec_launches(Decoder *d, int n) { d->spec_launches = n < 1 ? 1 : n; }

const void *dec_coef_ptr(Decoder *d, size_t *bytes) { *bytes = (size_t)d->nblocks_cap * 128; return d->d_coef; }

static int ensure(Decoder *d, size_t scan_len, const Geom &g, int restart_interval) {
    if (restart_interval > 0) {
        const size_t need = ((size_t)g.mcux * g.mcuy + restart_interval - 1) / restart_interval + 2;
        if (need > d->bnd_cap) {
            cudaFree(d->d_bnd); d->d_bnd = nullptr; d->bnd_cap = 0;
            DCK(cudaMalloc(&d->d_bnd, (need + need / 4) * 4));
            d->bnd_cap = need + need / 4;
        }
    }
    if (scan_len + 256 > d->scan_cap) {
        cudaFree(d->d_scan); cudaFree(d->d_u); d->d_scan = d->d_u = nullptr; d->scan_cap = 0;
        const size_t cap = scan_len + scan_len / 4 + 4096;
        DCK(cudaMalloc(&d->d_scan, cap));
        DCK(cudaMalloc(&d->d_u, cap));
        d->scan_cap = cap;
    }
    const size_t nsub = (scan_len * 8 + DEC_SUB_BITS - 1) / DEC_SUB_BITS + 256;
    if (nsub > d->nsub_cap) {
        cudaFree(d->d_st_in); cudaFree(d->d_st_out); cudaFree(d->d_nblk); cudaFree(d->d_blk_start); cudaFree(d->d_done);
        d->d_st_in = d->d_st_out = nullptr; d->d_nblk = d->d_blk_start = nullptr; d->d_done = nullptr; d->nsub_cap = 0;
        const size_t cap = nsub + nsub / 4;
        DCK(cudaMalloc(&d->d_st_in, cap * 8));
        DCK(cudaMalloc(&d->d_st_out, cap * 8));
        DCK(cudaMalloc(&d->d_nblk, (cap + 1) * 4));
        DCK(cudaMalloc(&d->d_blk_start, (cap + 1) * 4));
        DCK(cudaMalloc(&d->d_done, cap / 256 + 64));
        d->nsub_cap = cap;
    }
    // descriptor arrays: destuff chunks (4 KB), nblk scan chunks (2048), dc scan chunks (1024 blocks) x 3
    const size_t nd = std::max(std::max(scan_len / 4096, d->nsub_cap / 2048), (size_t)g.nblocks / 1024) + 8;
    if (nd > d->desc_cap) {
        cudaFree(d->d_desc); d->d_desc = nullptr; d->desc_cap = 0;
        DCK(cudaMalloc(&d->d_desc, nd * 5 * 8));
        d->desc_cap = nd;
    }
    const size_t pl = (size_t)g.mcux * 8 * g.hs * g.mcuy * 8 * g.vs + 2 * (size_t)g.mcux * 8 * g.mcuy * 8 + 256;
    if (pl > d->planes_cap) {
        cudaFree(d->d_planes); d->d_planes = nullptr; d->planes_cap = 0;
        DCK(cudaMalloc(&d->d_planes, pl));
        d->planes_cap = pl;
    }
    return B2J_OK;
}

int dec_run(Decoder *d, const uint8_t *jpg, size_t len, const JpegInfo &info, const Geom &g, uint8_t *d_bgr, size_t step,
            bool gray_out, cudaStream_t s, b2j_timings *tm, uint64_t *launches, bool careful, const uint8_t *d_scan_src,
            int scale) {
    const int rst = info.restart_interval;   // MCUs per restart interval (0: none)
    if (rst && info.scan_len >= 0xFFFFFFF0ull) { snprintf(d->err, d->errlen, "restart-marker scans of 4 GB and more are not supported"); return B2J_EFORMAT; }
    if (g.nblocks > d->nblocks_cap) { snprintf(d->err, d->errlen, "image exceeds the context's size"); return B2J_ESIZE; }
    if ((!d_scan_src && info.scan_offset + info.scan_len > len) || info.scan_len == 0) return B2J_EFORMAT;
    int rc = ensure(d, info.scan_len, g, rst);
    if (rc) return rc;
    const size_t n = info.scan_len;
    const size_t nsub_max = (n * 8 + DEC_SUB_BITS - 1) / DEC_SUB_BITS;
    const int hv = g.hs * g.vs;   // luma blocks per MCU (gray: 1 of 1)
    if (tm) cudaEventRecord(d->ev[0], s);
    // h_tb / h_flag are rewritten by the host below: a previous decode on this decoder must have drained first
    if (d->in_flight) { DCK(cudaStreamSynchronize(d->last_stream)); d->in_flight = false; }
    if (dec_build_tables(info, d->h_tb) != B2J_OK) { snprintf(d->err, d->errlen, "invalid Huffman table"); return B2J_EFORMAT; }
    d->last_stream = s;
    d->in_flight = true;
    DCK(cudaMemcpyAsync(d->d_tb, d->h_tb, dec_tables_size(), cudaMemcpyHostToDevice, s));
    DCK(cudaMemsetAsync(d->d_ctrl, 0, sizeof(DecCtrl), s));
    DCK(cudaMemsetAsync(d->d_desc, 0, d->desc_cap * 5 * 8, s));
    DCK(cudaMemsetAsync(d->d_nblk, 0, (nsub_max + 1) * 4, s));
    DCK(cudaMemsetAsync(d->d_done, 0, nsub_max / 256 + 64, s));

    // ---- self-synchronisation: launches of 8 in-CTA rounds until no end state moves.
    // Speculative mode (default): a fixed number of launches back to back, the "still moving" flag of the last one is
    // fetched asynchronously and looked at in dec_check -- no host round trip inside the decode, so several decoders
    // on different streams overlap. Streams with long synchronisation distances (about 200+ bits per block: blocks
    // rarely end with EOB) and retries take the careful mode: the host looks at the flag after every launch.
    const int DEC_SPEC_LAUNCHES = d->spec_launches;
    const bool spec = !careful && (double)n * 8.0 / (double)g.nblocks < 200.0;
    d->speculated = spec;
    d->h_flag[2] = 0;

    // ---- front end, pipelined: the scan goes up in pieces on its own stream; every piece is de-stuffed as soon as it
    // has landed and the first synchronisation pass runs on the decoder chunks whose bytes are complete, so most of
    // that pass hides behind the upload (large scans, speculative mode).
    const uint8_t *scan_in = d_scan_src ? d_scan_src : d->d_scan;
    const int nch = destuff_chunks(scan_in, n);   // d_scan is 256-byte aligned: pieces below fall on chunk borders
    // restart markers: one piece (a marker's two bytes may straddle pieces: k_destuff looks one byte ahead)
    const int npieces = (spec && n >= (16u << 20) && !rst && !d_scan_src) ? 8 : 1;   // fewer, larger pieces: a piece should fill the GPU
    uint32_t *bnd = rst ? d->d_bnd : nullptr;
    const uint32_t *nmark = rst ? &d->d_ctrl->nmark : nullptr;
    const size_t piece = ((n + npieces - 1) / npieces + DS_CHUNK - 1) & ~(size_t)(DS_CHUNK - 1);
    DCK(cudaEventRecord(d->ev_up[32], s));                       // the scan buffer is free once earlier work on s is done
    DCK(cudaStreamWaitEvent(d->up_stream, d->ev_up[32], 0));
    for (int j = 0; j < npieces; j++) {
        const size_t b0 = std::min(n, (size_t)j * piece), b1 = std::min(n, b0 + piece);
        if (b1 > b0 && !d_scan_src) {
            if (d->upload) {
                const int urc = d->upload(d->upload_user, d->d_scan + b0, jpg + info.scan_offset + b0, b1 - b0, d->up_stream);
                if (urc) return urc;
            } else {
                DCK(cudaMemcpyAsync(d->d_scan + b0, jpg + info.scan_offset + b0, b1 - b0, cudaMemcpyHostToDevice, d->up_stream));
            }
        }
        DCK(cudaEventRecord(d->ev_up[j], d->up_stream));
        DCK(cudaStreamWaitEvent(s, d->ev_up[j], 0));
        const int c0 = (int)(b0 / DS_CHUNK), c1 = j == npieces - 1 ? nch : (int)(b1 / DS_CHUNK);
        if (c1 > c0) {
            DCK(launch_destuff(scan_in, n, d->d_u, d->d_desc, &d->d_ctrl->dticket[j], c0, c1, &d->d_ctrl->u_len, &d->d_ctrl->avail,
                               bnd, (uint32_t)d->bnd_cap, &d->d_ctrl->nmark, &d->d_ctrl->err, s));
            if (launches) (*launches)++;
        }
        if (npieces > 1 && j < npieces - 1) {
            DCK(launch_dec_sync(d->d_u, &d->d_ctrl->avail, d->d_tb, d->d_st_in, d->d_st_out, d->d_nblk, g.bpm, hv, 8, 1, d->d_done,
                                &d->d_ctrl->changed, (b1 * 8 + DEC_SUB_BITS - 1) / DEC_SUB_BITS, bnd, nmark, nullptr, s));
            if (launches) (*launches)++;
        }
    }
    if (tm) cudaEventRecord(d->ev[1], s);
    int rounds = 0;
    if (spec) {
        const int nl = npieces > 1 ? std::max(1, DEC_SPEC_LAUNCHES - 1) : DEC_SPEC_LAUNCHES;
        uint32_t *flag = &d->d_ctrl->changed, *prev = nullptr;
        for (; rounds < nl; rounds++) {
            // a launch whose predecessor in this loop moved nothing returns at once (its own flag stays 0)
            flag = (rounds & 1) ? &d->d_ctrl->changed_alt : &d->d_ctrl->changed;
            DCK(cudaMemsetAsync(flag, 0, 4, s));
            DCK(launch_dec_sync(d->d_u, &d->d_ctrl->u_len, d->d_tb, d->d_st_in, d->d_st_out, d->d_nblk, g.bpm, hv, 8, 0, d->d_done,
                                flag, nsub_max, bnd, nmark, prev, s));
            prev = flag;
            if (launches) (*launches)++;
        }
        DCK(cudaMemcpyAsync(&d->h_flag[2], flag, 4, cudaMemcpyDeviceToHost, s));
        rounds--;
    } else {
        // long synchronisation distances / checked retry: one pass per launch, groups of subsequences per thread
        // (k_dec_sync_long); the host looks at the "an end state moved" flag after every launch
        // group length: a correction travels one group per launch and every launch is a pass over the stream, so streams
        // that practically never synchronise on their own (200+ bits per block) take long groups; the retry of an
        // ordinary stream keeps them short (more threads, few groups still moving after the second launch)
        const bool hard = (double)n * 8.0 / (double)g.nblocks >= 200.0;
        const int group = d->long_group > 0 ? d->long_group : (hard ? 32 : 8);
        for (;; rounds++) {
            if (rounds >= 65536) { snprintf(d->err, d->errlen, "Huffman synchronisation did not converge"); return B2J_EINTERNAL; }
            DCK(cudaMemsetAsync(&d->d_ctrl->changed, 0, 4, s));
            DCK(launch_dec_sync_long(d->d_u, &d->d_ctrl->u_len, d->d_tb, d->d_st_in, d->d_st_out, d->d_nblk, g.bpm, hv, rounds == 0, group,
                                     &d->d_ctrl->changed, nsub_max, bnd, nmark, s));
            if (launches) (*launches)++;
            if (rounds == 0) continue;  // the first launch always moves states
            DCK(cudaMemcpyAsync(d->h_flag, &d->d_ctrl->changed, 4, cudaMemcpyDeviceToHost, s));
            DCK(cudaStreamSynchronize(s));
            if (d->h_flag[0] == 0) break;
        }
    }
    d->last_rounds = rounds + 1;
    if (getenv("B2J_DEC_VERBOSE")) fprintf(stderr, "[b2j decode] %s synchronisation: %d launches, scan %zu bytes, %.1f bits/block\n", spec ? "scheduled" : "checked", d->last_rounds, n, (double)n * 8.0 / (double)g.nblocks);
    if (tm) cudaEventRecord(d->ev[2], s);
    DCK(launch_scan_u32(d->d_nblk, d->d_blk_start, nsub_max, d->d_desc + d->desc_cap, &d->d_ctrl->ticket[1], &d->d_ctrl->err, s));
    DCK(launch_dec_write(d->d_u, &d->d_ctrl->u_len, d->d_tb, d->d_st_out, d->d_blk_start, g.bpm, hv, d->d_coef, d->d_dc, (uint32_t)g.nblocks,
                         &d->d_ctrl->err, nsub_max, bnd, nmark, s));
    DCK(launch_dc_scan(d->d_dc, g, gray_out ? 1 : g.nc, d->d_desc + 2 * d->desc_cap, &d->d_ctrl->ticket[2], d->desc_cap,
                       &d->d_ctrl->err, s));
    if (tm) cudaEventRecord(d->ev[3], s);
    if (scale > 1) {   // reduced size: the scaled IDCT (gray: straight into the caller's image), colour on the scaled view
        uint8_t *py = d->d_planes;
        uint8_t *pcb = py + (((size_t)g.mcux * 8 * g.hs * g.mcuy * 8 * g.vs + 63) & ~(size_t)63);
        uint8_t *pcr = pcb + (((size_t)g.mcux * 8 * g.mcuy * 8 + 63) & ~(size_t)63);
        const DecScale sc = dec_scale_setup(g, scale);
        DCK(launch_idct_scaled(d->d_coef, d->d_dc, g, sc, d->d_tb, gray_out ? d_bgr : py, pcb, pcr, gray_out, step, rst, s));
        if (tm) cudaEventRecord(d->ev[4], s);
        if (!gray_out) DCK(launch_upcolor(py, pcb, pcr, sc.view, d_bgr, step, s));
        if (tm) cudaEventRecord(d->ev[5], s);
        if (launches) (*launches) += gray_out ? 4 : 5;
    } else if (gray_out) {   // Y straight from the IDCT into the caller's image: no planes, no colour pass (dec_color stays 0)
        DCK(launch_idct_gray(d->d_coef, d->d_dc, g, d->d_tb, d_bgr, step, rst, s));
        if (tm) { cudaEventRecord(d->ev[4], s); cudaEventRecord(d->ev[5], s); }
        if (launches) (*launches) += 4;
    } else {
        uint8_t *py = d->d_planes;
        uint8_t *pcb = py + (((size_t)g.mcux * 8 * g.hs * g.mcuy * 8 * g.vs + 63) & ~(size_t)63);
        uint8_t *pcr = pcb + (((size_t)g.mcux * 8 * g.mcuy * 8 + 63) & ~(size_t)63);
        DCK(launch_idct(d->d_coef, d->d_dc, g, d->d_tb, py, pcb, pcr, rst, s));
        if (tm) cudaEventRecord(d->ev[4], s);
        DCK(launch_upcolor(py, pcb, pcr, g, d_bgr, step, s));
        if (tm) cudaEventRecord(d->ev[5], s);
        if (launches) (*launches) += 5;
    }
    if (tm) {
        DCK(cudaStreamSynchronize(s));
        cudaEventElapsedTime(&tm->dec_parse, d->ev[0], d->ev[1]);
        cudaEventElapsedTime(&tm->dec_sync, d->ev[1], d->ev[2]);
        cudaEventElapsedTime(&tm->dec_write, d->ev[2], d->ev[3]);
        cudaEventElapsedTime(&tm->dec_idct, d->ev[3], d->ev[4]);
        cudaEventElapsedTime(&tm->dec_color, d->ev[4], d->ev[5]);
        cudaEventElapsedTime(&tm->total, d->ev[0], d->ev[5]);
    }
    return B2J_OK;
}

int dec_run_progressive(Decoder *d, const uint8_t *jpg, size_t len, const ProgInfo &info, const Geom &g, uint8_t *d_bgr,
                        size_t step, bool gray_out, cudaStream_t s, uint64_t *launches, int scale) {
    if (g.nblocks > d->nblocks_cap) { snprintf(d->err, d->errlen, "image exceeds the context's size"); return B2J_ESIZE; }
    int rc = ensure(d, 4096, g, 0);
    if (rc) return rc;
    if (d->in_flight) { DCK(cudaStreamSynchronize(d->last_stream)); d->in_flight = false; }
    d->speculated = false;
    d->last_stream = s;
    DCK(cudaMemsetAsync(&d->d_ctrl->err, 0, 4, s));
    return dec_progressive(jpg, len, info, g, d->d_coef, d->d_tb, d->d_planes, d_bgr, step, gray_out, s, launches, d->err, d->errlen,
                           scale);
}

int dec_check(Decoder *d, char *err, size_t errlen) {
    if (!d) return B2J_OK;
    if (cudaMemcpyAsync(&d->h_flag[1], &d->d_ctrl->err, 4, cudaMemcpyDeviceToHost, d->last_stream) != cudaSuccess ||
        cudaStreamSynchronize(d->last_stream) != cudaSuccess) {
        snprintf(err, errlen, "%s in dec_check", cudaGetErrorString(cudaGetLastError()));
        return B2J_ECUDA;
    }
    d->in_flight = false;
    if (d->speculated && d->h_flag[2]) return DEC_RETRY;   // the fixed number of launches was not enough: run again, carefully
    if (d->h_flag[1]) { snprintf(err, errlen, "decoder consistency check failed (err=%u)", d->h_flag[1]); return B2J_EINTERNAL; }
    return B2J_OK;
}

}  // namespace b2j
