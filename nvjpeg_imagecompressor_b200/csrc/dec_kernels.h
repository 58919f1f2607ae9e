// dec_kernels.h -- launchers of the decode kernels (internal)
#pragma once
#include "common.cuh"
#include "dec.h"

namespace b2j {

constexpr int DEC_LUT_BITS = 10;
constexpr int DEC_SUB_BITS = 1024;

struct DecTables {                 // device copy, one per decode
    uint16_t lut[4][1 << DEC_LUT_BITS];  // (len << 8) | symbol for codes of length <= DEC_LUT_BITS, else 0
    int32_t maxcode[4][18];        // maxcode[l] = largest code of length l, -1 if none; [17] = sentinel
    int32_t valoff[4][17];         // valptr[l] - mincode[l]
    uint8_t vals[4][256];
    uint16_t q[2][64];             // dequantisation table, natural order
};
size_t dec_tables_size();
// host side (dec_parse.cpp); B2J_EFORMAT for a table with more codes than its lengths allow
int dec_build_tables(const JpegInfo &info, void *dst_host);

// Chunks [c0, c1) of the n-byte scan (DS_CHUNK bytes of the 16-byte aligned stream that contains `in`: destuff_chunks()
// of them in all); `ticket`: a zeroed counter per launch; *avail = bytes produced so far
// bnd != NULL (restart markers): FF Dn pairs are dropped too; bnd[j] = output offset where interval j + 1 begins,
// bnd[*nmark] = 0xFFFFFFFF (bnd_cap entries available)
constexpr int DS_CHUNK = 16384;
inline int destuff_chunks(const void *in, size_t n) { return (int)(((reinterpret_cast<uintptr_t>(in) & 15) + n + DS_CHUNK - 1) / DS_CHUNK); }
cudaError_t launch_destuff(const uint8_t *in, size_t n, uint8_t *out, uint64_t *desc, uint32_t *ticket, int c0, int c1,
                           uint64_t *out_len, uint64_t *avail, uint32_t *bnd, uint32_t bnd_cap, uint32_t *nmark, uint32_t *err,
                           cudaStream_t s);
// mode 0: whole stream present (*u_len final); mode 1: stream still arriving (*u_len = bytes so far), first pass of the
// complete chunks only. done[chunk] (zeroed per decode) marks chunks whose first pass has run. nsub: subsequences covered.
cudaError_t launch_dec_sync(const uint8_t *u, const uint64_t *u_len, const void *tb, uint64_t *st_in, uint64_t *st_out,
                            uint32_t *nblk, int bpm, int hv, int inner, int mode, uint8_t *done, uint32_t *changed,
                            size_t nsub, const uint32_t *bnd, const uint32_t *nmark, const uint32_t *skip_if_zero, cudaStream_t s);
// long synchronisation distances and the checked retry: one launch = one pass, groups of 8 subsequences per thread;
// first != 0: every group starts from the guess, else from its predecessor's last end state (skipped if unchanged)
cudaError_t launch_dec_sync_long(const uint8_t *u, const uint64_t *u_len, const void *tb, uint64_t *st_in, uint64_t *st_out,
                                 uint32_t *nblk, int bpm, int hv, int first, int group, uint32_t *changed, size_t nsub,
                                 const uint32_t *bnd, const uint32_t *nmark, cudaStream_t s);
cudaError_t launch_dec_write(const uint8_t *u, const uint64_t *u_len, const void *tb, const uint64_t *st_out,
                             const uint32_t *blk_start, int bpm, int hv, int16_t *coef, int16_t *dcarr, uint32_t nblocks,
                             uint32_t *err, size_t nsub_max, const uint32_t *bnd, const uint32_t *nmark, cudaStream_t s);
cudaError_t launch_scan_u32(const uint32_t *in, uint32_t *out, size_t n, uint64_t *desc, uint32_t *ticket, uint32_t *err,
                            cudaStream_t s);
// coef here = the compact DC array (one int16 per block); ncomp: the first ncomp components (1: luma only)
cudaError_t launch_dc_scan(int16_t *coef, const Geom &g, int ncomp, uint64_t *desc, uint32_t *ticket, size_t desc_stride,
                           uint32_t *err, cudaStream_t s);
// rst_mcus: restart interval in MCUs (0: none): DC predictors return to 0 at every interval start
cudaError_t launch_idct(const int16_t *coef, const int16_t *dcarr, const Geom &g, const void *tb, uint8_t *py, uint8_t *pcb,
                        uint8_t *pcr, int rst_mcus, cudaStream_t s);
// the luma blocks only, their samples stored straight into the caller's 8-bit image (gray output: libjpeg's
// JCS_GRAYSCALE, no upsampling or colour conversion); chroma blocks of a three-component file are skipped
cudaError_t launch_idct_gray(const int16_t *coef, const int16_t *dcarr, const Geom &g, const void *tb, uint8_t *gray, size_t step,
                             int rst_mcus, cudaStream_t s);
// halo_top / halo_bottom: the chroma planes hold one valid row above row 0 / below the last row (a strip of a larger
// image: the vertical filter of 4:2:0 / 4:4:0 then reads the neighbour strip's row instead of replicating the edge)
cudaError_t launch_upcolor(const uint8_t *py, const uint8_t *pcb, const uint8_t *pcr, const Geom &g, uint8_t *bgr, size_t step,
                           cudaStream_t s, int halo_top = 0, int halo_bottom = 0);

// ---- reduced-size decode (dec_scaled.cu): libjpeg's DCT scaling with scale_num = 1, scale_denom = 2 / 4 / 8 (jdmaster.c)
// Output W' x H' = ceil(W / denom) x ceil(H / denom). A luma block gives S x S samples (S = 8 / denom); a chroma block
// Sc x Sc, where Sc starts at S and doubles while it is below 8 and both (hs S) % (2 Sc) and (vs S) % (2 Sc) are 0
// (4:2:0: Sc = 2 S). The true chroma size is ceil(W Sc / (hs 8)) x ceil(H Sc / (vs 8)). Chroma reaches the output size
// through k_upcolor unchanged, on `view`: a Geom whose W / H are the output size, dw[1] / dh[1] the true chroma size, hs /
// vs the k_upcolor instantiation (hs S / Sc x vs S / Sc) and mcux the file's (the planes' pitches mcux 8 hs and mcux 8
// hold the scaled rows). jdsample.c turns its fancy filters off when Sc = 1: 4:2:2 and 4:4:0 at 1/8 replicate, which
// the IDCT does itself (rep) so that the view is 1 x 1.
inline int dec_scaled_size(int n, int denom) { return (n + denom - 1) / denom; }
struct DecScale {
    int S, Sc;      // output size of a luma / chroma block
    int rep;        // 0, or every chroma sample stored twice: 1 side by side (4:2:2 at 1/8), 2 one above the other (4:4:0)
    Geom view;
};
inline DecScale dec_scale_setup(const Geom &g, int denom) {
    DecScale d;
    d.S = 8 / denom;
    d.Sc = d.S;
    while (d.Sc < 8 && (g.hs * d.S) % (2 * d.Sc) == 0 && (g.vs * d.S) % (2 * d.Sc) == 0) d.Sc *= 2;
    int hx = g.hs * d.S / d.Sc, vx = g.vs * d.S / d.Sc;
    d.rep = 0;
    if (d.Sc == 1 && hx == 2 && vx == 1) { d.rep = 1; hx = 1; }
    if (d.Sc == 1 && hx == 1 && vx == 2) { d.rep = 2; vx = 1; }
    d.view = g;
    d.view.W = dec_scaled_size(g.W, denom);
    d.view.H = dec_scaled_size(g.H, denom);
    d.view.hs = hx; d.view.vs = vx;
    d.view.dw[0] = d.view.W; d.view.dh[0] = d.view.H;
    for (int c = 1; c < g.nc; c++) {
        d.view.dw[c] = (g.W * d.Sc + g.hs * 8 - 1) / (g.hs * 8);
        d.view.dh[c] = (g.H * d.Sc + g.vs * 8 - 1) / (g.vs * 8);
    }
    return d;
}
// gray: the luma blocks only, clipped into the caller's 8-bit image (py, pitch out_step); else Y into py (pitch
// mcux 8 view.hs) and Cb / Cr into pcb / pcr (pitch mcux 8), for launch_upcolor(py, pcb, pcr, sc.view, ...)
cudaError_t launch_idct_scaled(const int16_t *coef, const int16_t *dcarr, const Geom &g, const DecScale &sc, const void *tb,
                               uint8_t *py, uint8_t *pcb, uint8_t *pcr, bool gray, size_t out_step, int rst_mcus, cudaStream_t s);

// progressive files (dec_prog.cu): all scans into d_coef, then IDCT + upsampling; synchronises the stream before returning
// gray_out: 8-bit Y samples into d_bgr (launch_idct_gray) instead of IDCT + upsampling + colour conversion
// scale: 1, or the reduced-size back end (launch_idct_scaled) at 1 / scale
int dec_progressive(const uint8_t *jpg, size_t len, const ProgInfo &info, const Geom &g, int16_t *d_coef, void *d_tb,
                    uint8_t *d_planes, uint8_t *d_bgr, size_t step, bool gray_out, cudaStream_t s, uint64_t *launches,
                    char *err, size_t errlen, int scale = 1);

}  // namespace b2j
