// kernels.h -- host-callable launchers of the sm_100a kernels (internal to libb2jpeg.so)
#pragma once
#include "common.cuh"

namespace b2j {

// encode
int fdct_tm_max(int hs, int vs, int nc);   // MCUs per fdct tile (even); nc = components per image
// MCU rows [my0, my0+nrows) of the image `img` (img points at pixel row 0); coef_dump != NULL also writes coefficients
cudaError_t launch_fdct(const uint8_t *img, size_t step, const Geom &g, const QuantDev *qd, uint32_t *pool,
                        uint32_t *pool_count, uint32_t *ticket, TileRec *recs, uint32_t *hist, int do_hist, int my0, int nrows,
                        int16_t *coef_dump, cudaStream_t s);   // ticket: zeroed, one per launch
// xr != NULL: one-collective strip exchange (first MCU left to k_strip_merge, record fields filled)
// resolve != 0: also rewrite each tile's three raw-DC tokens in `pool` as final DC-difference tokens
cudaError_t launch_dc_edge_hist(const TileRec *recs, const Geom &g, const int16_t *pred_in, uint32_t *hist,
                                int16_t *last_dc, int do_hist, uint32_t *pool, int resolve, StripRecord *xr, int rst_tiles,
                                cudaStream_t s);
// restart_interval != 0: DRI marker (MCUs per interval) between the DHTs and SOS
// nc == 1 (gray): only DC0/AC0 are built and emitted, with the one-component DQT / SOF0 / SOS
cudaError_t launch_tables(const uint32_t *hist, int optimize, HuffDev *huff, const QuantDev *qd, int full_w, int full_h,
                          int hs, int vs, int nc, uint8_t *out, int emit_header, int restart_interval, uint32_t *err_out, cudaStream_t s);
// restart intervals of rst_tiles tiles (whole MCU rows): every interval but the last gets 1-padding to a byte boundary
// and its RSTn marker appended to its last tile's bits (run between k_pack and the tile scan)
cudaError_t launch_rst_pad(uint32_t *slots, uint32_t *tile_bits, int ntiles, int rst_tiles, cudaStream_t s);
// small_buffers != 0 (tests): the per-warp bit buffers pretend to hold 24 words, forcing the overflow path
cudaError_t launch_pack(const uint32_t *pool, const TileRec *recs, const Geom &g, const HuffDev *huff,
                        uint32_t *slots, uint32_t *tile_bits, int small_buffers, cudaStream_t s);
// desc: scan_desc_count(ntiles) zeroed look-back descriptors; ticket: zeroed. Also writes, for every k_stuff chunk
// c < nchunk_cap that starts inside the strip, the tile that holds its first bit (k_stuff starts there: no search)
int scan_desc_count(int ntiles);
cudaError_t launch_scan_tiles(const uint32_t *tile_bits, int ntiles, uint64_t *tile_off, const uint32_t *slots,
                              uint64_t *strip_bits, uint64_t *desc, uint32_t *ticket, uint32_t *chunk_tile,
                              uint32_t nchunk_cap, uint32_t *err, cudaStream_t s);
struct StuffArgs {
    const uint32_t *slots;
    const uint32_t *tile_bits;
    const uint64_t *tile_off;   // [ntiles+1]
    const uint32_t *chunk_tile; // tile holding bit c * 8 * STUFF_CHUNK of the strip's bit string (from the tile scan)
    int ntiles;
    const int *seam;            // device: [0] skip = leading bits owned by the previous strip's last byte,
                                //         [1] ext ^ 0xFF, ext = next strip's first 8 bits (0xFF: pad with ones)
    int append_eoi;
    int rst_tiles;              // tiles per restart interval (0: none): the markers' 0xFF bytes are not stuffed
    const HuffDev *huff;        // hdr_len
    uint8_t *out;
    size_t cap;
    uint64_t *desc;             // look-back descriptors (zeroed)
    uint32_t *ticket;           // zeroed
    uint64_t *out_len;
    uint32_t *err;
};
cudaError_t launch_stuff(const StuffArgs &a, int grid, cudaStream_t s);
// seam[0..1] from host scalars, or from the all-gathered per-strip (bit count, first 32 bits) table on the device
cudaError_t launch_set_seam(int *seam, int skip, int ext, cudaStream_t s);
cudaError_t launch_seam_from_bits(int *seam, const int64_t *bits_all, int rank, int world, cudaStream_t s);
// one-collective strip exchange: rec = the all-gathered records [world]
// flags != NULL: wait (bounded) until flags[0..world) == seq before reading rec (peer-memory exchange)
cudaError_t launch_strip_merge(const StripRecord *rec, int rank, int world, uint32_t *hist, uint32_t *pool,
                               const TileRec *recs, const uint32_t *flags, uint32_t seq, unsigned long long timeout_ns,
                               uint32_t *err, cudaStream_t s);
// store this strip's record into every rank's arena (peers[world], device array) and raise the flags
cudaError_t launch_strip_push(const StripRecord *mine, XchgArena *const *peers, int rank, int world, uint32_t seq, cudaStream_t s);
cudaError_t launch_strip_seam(const StripRecord *rec, int rank, int world, HuffDev *huff, int drop_header, int *seam,
                              const uint64_t *strip_bits, uint32_t *err, cudaStream_t s);

// decode
struct DecArgs;
// metrics
cudaError_t launch_diff_psnr(const uint8_t *a, const uint8_t *b, size_t n, int mode, uint8_t *out, uint64_t *ssd,
                             cudaStream_t s);

}  // namespace b2j
