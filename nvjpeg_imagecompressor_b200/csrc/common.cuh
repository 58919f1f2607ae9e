// common.cuh -- shared device/host declarations of the B200 JPEG engine (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace b2j {

// ---- geometry of one image / MCU-row strip (libjpeg jcmaster.c per_scan_setup) -------------------------
struct Geom {
    int W, H;          // pixels
    int hs, vs;        // luma sampling factors; chroma is 1x1 (gray: 1x1)
    int mcux, mcuy;    // MCU grid
    int bpm;           // blocks per MCU = hs*vs + 2 (gray: 1)
    int wib[3], hib[3];// real blocks per component (width/height in blocks)
    int dh[3];         // true downsampled height in samples
    int dw[3];         // true downsampled width in samples
    int tm;            // MCUs per fdct tile (even)
    int tiles_x;       // fdct tiles per MCU row
    int nblocks;       // mcux*mcuy*bpm, scan order
    int ntiles;        // fdct/pack tiles = tiles_x * mcuy
    int nc;            // components per image: 3 (Y, Cb, Cr) or 1 (gray: one non-interleaved scan, an MCU is one block)
};

// One token per coded coefficient / EOB / DC difference:
//   [27:26] number of ZRL (0xF0) symbols that precede it (zero run >> 4)   [25:22] zero run & 15
//   [21:18] size (bits of |value|)      [17:16] (tcode + zero run) & 3, tcode: 0 AC luma, 1 AC chroma, 2 DC luma, 3 DC chroma
//   [15:0]  value bits (already masked to `size` bits)
// Bits [25:16] index the symbol: k_fdct's histogram bins and k_pack's code tables use this order. It is chosen for
// the shared-memory banks of those tables (32 lanes look up 32 different tokens): the bank is (size & 7) << 2 |
// (tcode + run) & 3, so the common symbols -- sizes 0..7 of runs 0..3 of one table -- sit in 32 different banks. The run
// enters the table field for free: the run counter of k_fdct's walk advances both fields with one add (tcode <= 1 for
// the AC tables and runs <= 62 keep that sum inside bits [21:16]; stage C masks the size field).
// Huffman tables elsewhere are numbered 0 DC0, 1 AC0, 2 DC1, 3 AC1 (HuffDev, histograms).
// TOK_RAWDC: DC of a block whose predecessor lives in the previous tile; [17:16] tcode, [19:18] component, [15:0] the
// quantised DC itself (k_dc_edge_hist rewrites it as a difference token).
constexpr uint32_t TOK_RAWDC = 1u << 28;
constexpr uint32_t TOK_RUN_STEP = (1u << 22) + (1u << 16);   // one more zero coefficient: run field and table field
__host__ __device__ constexpr uint32_t tcode_of(uint32_t table) { return (table & 1u) ? (table >> 1) : 2u + (table >> 1); }
__host__ __device__ constexpr uint32_t table_of(uint32_t tcode) { return tcode < 2u ? 2u * tcode + 1u : 2u * (tcode - 2u); }
__host__ __device__ constexpr uint32_t tok_bin(uint32_t table, uint32_t sym) {   // bin of (Huffman table, JPEG symbol)
    return (table & 1u) ? ((((sym >> 4) & 15u) << 6) | ((sym & 15u) << 2) | ((tcode_of(table) + (sym >> 4)) & 3u))
                        : (((sym & 15u) << 2) | tcode_of(table));
}
__host__ __device__ constexpr uint32_t bin_table(uint32_t bin) { return table_of(((bin & 3u) - (bin >> 6)) & 3u); }
__host__ __device__ constexpr uint32_t bin_symbol(uint32_t bin) {   // JPEG symbol of a bin (DC bins carry no run)
    return (bin_table(bin) & 1u) ? (((bin >> 6) << 4) | ((bin >> 2) & 15u)) : ((bin >> 2) & 15u);
}
__host__ __device__ constexpr uint32_t tok_dc(uint32_t table, uint32_t size, uint32_t vbits) { return (tcode_of(table) << 16) | (size << 18) | vbits; }
struct TileRec {                               // one per fdct tile (<= 256 blocks, one MCU-row segment)
    uint32_t base, count;                      // token run in the pool
    int16_t first_dc[3], last_dc[3];           // DCs of the tile's first / last MCU (last Y block, Cb, Cr; gray: [0] only)
    uint16_t pos_cb, pos_cr;                   // run offsets of the first MCU's Cb / Cr DC tokens (Y: offset 0)
};

// What the strips of one image tell each other (multi-GPU encode, one all-gather of this record per image;
// include/b2jpeg.h: b2j_strip_record). The DC symbols of the strip's first MCU are NOT in hist: their predictors live
// in the previous strip, every rank derives them for every strip from first_dc / last_dc after the exchange.
struct StripRecord {
    uint32_t hist[4 * 257];   // symbol counts of this strip: DC0, AC0, DC1, AC1
    int16_t first_dc[4];      // quantised DC of the strip's first Y, Cb, Cr blocks
    int16_t last_dc[4];       // ... of its last Y, Cb, Cr blocks
    uint32_t tok[8];          // first tokens of the strip (raw-DC tokens unresolved): the next 8+ bits after the seam
    uint32_t ntok;
    uint32_t pad[3];
};
static_assert(sizeof(StripRecord) == 4176, "b2j_strip_record layout");

// Peer-memory exchange of the records (GPUs of one node): every rank owns one arena; peers store their record of
// image `seq` straight into set (seq % SETS), slot [their rank], over NVLink and then raise flags[set][rank] = seq.
constexpr int XCHG_SETS = 4;                   // images in flight before a slot is reused (2 would do: DESIGN.md 5)
constexpr int XCHG_MAX_WORLD = 16;
struct XchgArena {
    uint32_t flags[XCHG_SETS][XCHG_MAX_WORLD];   // [set][sender] = sequence number of the image whose record is in place
    StripRecord rec[XCHG_SETS][XCHG_MAX_WORLD];
};

constexpr int PACK_BLOCKS = 256;               // blocks per pack tile (= fdct tile capacity)
constexpr int SLOT_WORDS = PACK_BLOCKS * 52 + 4; // worst case 64 coefs * 26 bits = 52 words per block, + pad/RSTn bits of an interval end
#ifndef B2J_STUFF_THREADS
#define B2J_STUFF_THREADS 256
#endif
#ifndef B2J_STUFF_CTAS
#define B2J_STUFF_CTAS 4
#endif
#ifndef B2J_STUFF_PIECES
#define B2J_STUFF_PIECES 4
#endif
constexpr int STUFF_THREADS = B2J_STUFF_THREADS;
constexpr int STUFF_CTAS = B2J_STUFF_CTAS;     // resident CTAs per SM: the chunk pipeline is latency bound (ticket, look-back)
constexpr int STUFF_PIECES = B2J_STUFF_PIECES;  // 16-byte pieces per thread and chunk (strided by STUFF_THREADS * 16)
constexpr int STUFF_BPT = 16 * STUFF_PIECES;    // unstuffed bytes per thread and chunk
constexpr int STUFF_CHUNK = STUFF_THREADS * STUFF_BPT; // unstuffed bytes per stuff chunk

// ---- zig-zag ------------------------------------------------------------------------------------------
__host__ __device__ constexpr int zigzag_nat(int k) {
    constexpr int z[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                           41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                           30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
    return z[k];
}

// run-time index variant (one table in constant memory instead of a compile-time select chain)
__device__ __constant__ const uint8_t c_zigzag_nat[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                                                           41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                                                           30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
__device__ __forceinline__ int zigzag_nat_rt(int k) { return c_zigzag_nat[k]; }

// ---- device-side tables -------------------------------------------------------------------------------
struct QuantDev {          // forward: q = low half of fma(c, finv, 1.5 * 2^35), finv = 4096 (1 + 2^-20) / (8 q); natural order; [0] luma, [1] chroma
    float finv[2][64];
    uint16_t q[2][64];     // natural order quant values (dequantisation + DQT marker)
};

struct HuffDev {           // produced by k_tables
    uint32_t enc[4][256];  // (code << 8) | length, index: DC0, AC0, DC1, AC1
    uint8_t bits[4][17];
    uint8_t vals[4][256];
    uint32_t nsym[4];
    uint32_t hdr_len;      // bytes of SOI..SOS written at the start of the output buffer
    uint32_t err;
};

// look-back descriptor: [63:62] status, [61:0] value
constexpr uint64_t LB_AGG = 1ull << 62, LB_INC = 2ull << 62, LB_MASK = (1ull << 62) - 1;

// ---- small device helpers -----------------------------------------------------------------------------
// Programmatic dependent launch: kernels launched with launch_pdl() may become resident while their predecessor in
// the stream still runs; nothing the predecessor wrote may be touched before pdl_wait(). Small predecessors call
// pdl_trigger() first thing so that the next kernel's CTAs set up (shared-memory clears, tables) under them.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
#ifdef __CUDACC__
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}
#endif

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// 1-D TMA bulk copy global -> shared, completion on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, unsigned bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, unsigned parity) {
    uint32_t ok;
    uint32_t a = smem_u32(bar);
    do {
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                     : "=r"(ok)
                     : "r"(a), "r"(parity)
                     : "memory");
    } while (!ok);
}

__device__ __forceinline__ uint4 ld_nc_v4(const void *p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ void st_na_v4(void *p, uint4 v) {
    asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w)
                 : "memory");
}
__device__ __forceinline__ uint64_t ld_volatile_u64(const uint64_t *p) {
    uint64_t v;
    asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_volatile_u64(uint64_t *p, uint64_t v) {
    asm volatile("st.volatile.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// Decoupled look-back over 64-bit descriptors; executed by ONE full warp. Chunk ids must be handed out in
// launch order (atomic ticket) so every predecessor is resident or finished. Returns the exclusive prefix.
__device__ __forceinline__ uint64_t lookback_exclusive(uint64_t *desc, int id, uint64_t local, uint32_t *err) {
    const int lane = threadIdx.x & 31;
    if (id == 0) {
        if (lane == 0) st_volatile_u64(&desc[0], LB_INC | local);
        return 0;
    }
    if (lane == 0) st_volatile_u64(&desc[id], LB_AGG | local);
    uint64_t prefix = 0;
    int j = id - 1;
    for (;;) {
        int idx = j - lane;
        uint64_t d = LB_INC;
        if (idx >= 0) {
            unsigned spins = 0;
            d = ld_volatile_u64(&desc[idx]);
            while ((d >> 62) == 0) {
                __nanosleep(20);
                d = ld_volatile_u64(&desc[idx]);
                if (++spins > (1u << 22)) { *err = 1; d = LB_INC; break; }  // never hang the GPU
            }
        }
        unsigned inc = __ballot_sync(0xffffffffu, (d >> 62) == 2);
        int first = inc ? (__ffs(inc) - 1) : 32;
        uint64_t v = (lane <= first) ? (d & LB_MASK) : 0;
#pragma unroll
        for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        prefix += v;
        if (inc) break;
        j -= 32;
    }
    if (lane == 0) st_volatile_u64(&desc[id], LB_INC | ((prefix + local) & LB_MASK));
    return prefix;
}

}  // namespace b2j
