// dec_kernels.cu -- the decode path: de-stuff, self-synchronising parallel Huffman decode, DC prefix sums,
// islow IDCT, fancy upsampling + YCbCr->BGR with an interleaved store.
//
// Replaces nvjpegDecodeJpegHost / TransferToDevice / Device (reference call sites ImageCompressorImpl.cu:364-366)
// and the planar->interleaved CPU loop getCVImageOnCPU (:184-232; the dead combineChannels kernel :171-182).
// Arithmetic follows libjpeg-turbo jdhuff.c / jidctint.c / jdsample.c / jdcolor.c as restated in SURVEY.md
// Appendix A.9, pixel-exactly. The stream has no restart markers, so the Huffman stage is the self-synchronising
// scheme of Weissenberger & Schmidt (ICPP'18): every thread decodes a fixed 1024-bit subsequence from a guessed
// state, then re-decodes from its predecessor's end state until the states stop changing (SURVEY.md App. D).
#include <algorithm>
#include <atomic>

#include "common.cuh"
#include "dec.h"
#include "dec_idct.cuh"
#include "dec_kernels.h"

namespace b2j {

// ------------------------------------------------------------------------------------------------------
// k_destuff: drop the 0x00 that follows every 0xFF. Persistent CTAs take 16 KB chunks by ticket: every thread loads four
// 16-byte vectors (piece p of all threads, then piece p + 1: the stream order), finds the dropped bytes with byte-lane
// arithmetic on the words, the kept-byte counts are scanned across the CTA and chained by a decoupled look-back, the
// kept bytes are compacted word by word with a 16-entry table of PRMT selectors into a zeroed staging buffer and
// copied out as 16-byte vectors. Output is padded with 0xFF bytes (1-bits).
// The input may start at any address: the chunk grid is laid over the 16-byte aligned stream that begins up to 15
// bytes earlier (bytes outside [in, in + n) count as absent), so every load is an aligned vector.
// One launch handles the chunks [c0, c1) of the scan (the bytes before them are already there: a byte only looks at
// its predecessor), so the scan can be de-stuffed piece by piece while it is still being uploaded; look-back
// descriptors carry over, `ticket` is a fresh counter per launch, *avail = bytes produced up to the end of the launch.
// RST (streams with restart markers, jdmarker.c read_restart_marker): the two bytes of every FF Dn are dropped as well
// and the output offset where the next interval begins goes to bnd[j], j = ordinal of the marker (the look-back
// carries the marker count in the upper bits of its sums); bnd[number of markers] = 0xFFFFFFFF closes the list.
// So is every 0xFF followed by 0xFF: the fill bytes a marker may have in front of it (T.81 B.1.1.2; an 0xFF of
// entropy data is always followed by a stuffed zero). Fill before the terminating marker is cut off by the parser.
constexpr int DS_MK_SHIFT = 38;   // look-back value: kept bytes | markers << 38
constexpr int DS_THREADS = 256, DS_NP = 4;
static_assert(DS_THREADS * 16 * DS_NP == DS_CHUNK, "chunk = four 16-byte pieces per thread");
constexpr int DS_OUT_WORDS = (DS_CHUNK + 64) / 4;

// bit 7 of every byte lane: the byte is 0xFF / is 0x00
__device__ __forceinline__ uint32_t lanes_ff(uint32_t w) { return ((w & 0x7F7F7F7Fu) + 0x01010101u) & w & 0x80808080u; }
__device__ __forceinline__ uint32_t lanes_zero(uint32_t w) { return ~(((w & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | w) & 0x80808080u; }
// bits 7, 15, 23, 31 -> bits 0..3
__device__ __forceinline__ uint32_t lanes_to_bits(uint32_t m) { return ((m >> 7) * 0x01020408u) >> 24 & 15u; }

template <bool RST>
__global__ void __launch_bounds__(DS_THREADS)
k_destuff(const uint8_t *__restrict__ in, size_t n, uint8_t *__restrict__ out, uint64_t *__restrict__ desc,
          uint32_t *__restrict__ ticket, int c0, int c1, uint64_t *__restrict__ out_len, uint64_t *__restrict__ avail,
          uint32_t *__restrict__ bnd, uint32_t bnd_cap, uint32_t *__restrict__ nmark, uint32_t *__restrict__ err) {
    __shared__ int s_chunk;
    __shared__ uint32_t s_warp[DS_NP][DS_THREADS / 32];
    __shared__ uint64_t s_goff;
    __shared__ uint32_t s_lut[16];
    __shared__ __align__(16) uint32_t s_out32[DS_OUT_WORDS];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const uint32_t sbase = smem_u32(s_out32);
    const size_t lo = reinterpret_cast<uintptr_t>(in) & 15, hi = lo + n;   // the stream's bytes in the aligned stream
    const uint8_t *ina = in - lo;
    const int nchunks = (int)((hi + DS_CHUNK - 1) / DS_CHUNK);
    if (tid < 16) {   // PRMT selectors: the bytes of a word that are not dropped (bit i of tid: byte i is), in order, zero fill
        uint32_t sel = 0;
        int k = 0;
        for (int i = 0; i < 4; i++)
            if (!(tid & (1 << i))) sel |= (uint32_t)i << (4 * k++);
        for (; k < 4; k++) sel |= 4u << (4 * k);
        s_lut[tid] = sel;
    }
    for (int i = tid; i < DS_OUT_WORDS; i += DS_THREADS) s_out32[i] = 0;
    __syncthreads();
    for (;;) {
        if (tid == 0) s_chunk = c0 + (int)atomicAdd(ticket, 1u);
        __syncthreads();
        const int ch = s_chunk;
        if (ch >= c1) break;
        uint32_t x[DS_NP][4], keep[DS_NP], mark[DS_NP], cnt[DS_NP], inc[DS_NP];
#pragma unroll
        for (int p = 0; p < DS_NP; p++) {
            const size_t base = (size_t)ch * DS_CHUNK + (size_t)p * (DS_THREADS * 16) + (size_t)tid * 16;
            uint4 v = make_uint4(0, 0, 0, 0);
            uint32_t valid = 0;   // bit i: byte i of the piece belongs to the stream
            if (base < hi && base + 16 > lo) {
                v = *reinterpret_cast<const uint4 *>(ina + base);
                const uint32_t b0 = base < lo ? (uint32_t)(lo - base) : 0u, b1 = base + 16 > hi ? (uint32_t)(hi - base) : 16u;
                valid = ((1u << b1) - 1u) & ~((1u << b0) - 1u);
                if (valid != 0xFFFFu) {   // absent bytes read as zero
                    uint32_t *w = &v.x;
#pragma unroll
                    for (int q = 0; q < 4; q++) {
                        const uint32_t vb = (valid >> (4 * q)) & 15u;
                        w[q] &= ((vb * 0x00204081u) & 0x01010101u) * 0xFFu;
                    }
                }
            }
            x[p][0] = v.x; x[p][1] = v.y; x[p][2] = v.z; x[p][3] = v.w;
            // the byte before the piece / after it: the neighbour lane's, or one byte load at the warp's ends
            uint32_t prevb = __shfl_up_sync(0xffffffffu, v.w >> 24, 1);
            if (lane == 0) prevb = (base > lo && base - 1 < hi) ? ina[base - 1] : 0u;
            uint32_t nextb = 0;
            if (RST) {
                nextb = __shfl_down_sync(0xffffffffu, v.x & 0xFFu, 1);
                if (lane == 31) nextb = (base + 16 >= lo && base + 16 < hi) ? ina[base + 16] : 0u;
            }
            uint32_t ff[4], drop[4], sec[4] = {0, 0, 0, 0}, d0[4] = {0, 0, 0, 0};
#pragma unroll
            for (int q = 0; q < 4; q++) {
                ff[q] = lanes_ff(x[p][q]);
                if (RST) d0[q] = lanes_zero((x[p][q] & 0xF8F8F8F8u) ^ 0xD0D0D0D0u);   // bytes D0 .. D7
            }
            const uint32_t ffprev = prevb == 0xFFu ? 0x80000000u : 0u;
            const uint32_t d0next = (nextb & 0xF8u) == 0xD0u ? 0x80u : 0u, ffnext = nextb == 0xFFu ? 0x80u : 0u;
            uint32_t k16 = 0, m16 = 0;
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const uint32_t pf = __funnelshift_l(q ? ff[q - 1] : ffprev, ff[q], 8);          // the byte before is 0xFF
                drop[q] = lanes_zero(x[p][q]) & pf;
                if (RST) {
                    sec[q] = pf & d0[q];                                                        // second byte of FF Dn
                    const uint32_t nd = __funnelshift_r(d0[q], q < 3 ? d0[q + 1] : d0next, 8);  // the byte after is Dn
                    const uint32_t nf = __funnelshift_r(ff[q], q < 3 ? ff[q + 1] : ffnext, 8);  // the byte after is 0xFF
                    drop[q] |= sec[q] | (ff[q] & (nd | nf));                                    // ... and its first byte
                    m16 |= lanes_to_bits(sec[q]) << (4 * q);
                }
                k16 |= lanes_to_bits(drop[q] ^ 0x80808080u) << (4 * q);
            }
            // (absent bytes read as zero, so an 0xFF that ends the stream is data: a marker needs both of its bytes)
            keep[p] = k16 & valid;
            mark[p] = m16 & valid;
            cnt[p] = __popc(keep[p]) | (RST ? (uint32_t)__popc(mark[p]) << 16 : 0u);   // kept bytes | markers << 16
            inc[p] = cnt[p];
        }
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
#pragma unroll
            for (int p = 0; p < DS_NP; p++) {
                const uint32_t y = __shfl_up_sync(0xffffffffu, inc[p], o);
                if (lane >= o) inc[p] += y;
            }
        }
        if (lane == 31) {
#pragma unroll
            for (int p = 0; p < DS_NP; p++) s_warp[p][wid] = inc[p];
        }
        __syncthreads();
        uint32_t ex[DS_NP], total = 0;   // exclusive prefix in stream order (piece-major): kept bytes | markers << 16
#pragma unroll
        for (int p = 0; p < DS_NP; p++) {
            uint32_t wb = 0, tt = 0;
#pragma unroll
            for (int k = 0; k < DS_THREADS / 32; k++) {
                const uint32_t y = s_warp[p][k];
                if (k < wid) wb += y;
                tt += y;
            }
            ex[p] = total + wb + inc[p] - cnt[p];
            total += tt;
        }
        if (wid == 0) {   // the other warps compact meanwhile
            const uint64_t local = (uint64_t)(total & 0xFFFFu) | ((uint64_t)(total >> 16) << DS_MK_SHIFT);
            const uint64_t pre = lookback_exclusive(desc, ch, local, err);
            if (lane == 0) s_goff = pre;
        }
        // ---- the kept bytes of every word, compacted, OR-ed into the zeroed staging buffer at their chunk-local offset
#pragma unroll
        for (int p = 0; p < DS_NP; p++) {
            uint32_t o = ex[p] & 0xFFFFu;
            if (keep[p]) {
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    const uint32_t d4 = (~keep[p] >> (4 * q)) & 15u;
                    const uint32_t bytes = __byte_perm(x[p][q], 0u, s_lut[d4]);
                    const uint32_t bs = (o & 3u) * 8u, addr = sbase + (o & ~3u);
                    const uint32_t y0 = bytes << bs, y1 = __funnelshift_l(bytes, 0u, bs);
                    asm volatile("red.shared.or.b32 [%0], %1;" ::"r"(addr), "r"(y0) : "memory");
                    if (y1) asm volatile("red.shared.or.b32 [%0+4], %1;" ::"r"(addr), "r"(y1) : "memory");
                    o += 4u - __popc(d4);
                }
            }
        }
        __syncthreads();
        const uint64_t goff = s_goff & ((1ull << DS_MK_SHIFT) - 1);
        const uint32_t tkept = total & 0xFFFFu;
        uint8_t *dst = out + goff;
        {   // copy out: bytes up to the first 16-byte boundary and behind the last one singly, 16-byte vectors between
            const uint8_t *s_out = reinterpret_cast<const uint8_t *>(s_out32);
            const uint32_t head = min(tkept, (16u - (uint32_t)(reinterpret_cast<uintptr_t>(dst) & 15u)) & 15u);
            const uint32_t nvec = (tkept - head) >> 4, tail0 = head + 16u * nvec;
            if ((uint32_t)tid < head) dst[tid] = s_out[tid];
            if (tail0 + (uint32_t)tid < tkept) dst[tail0 + tid] = s_out[tail0 + tid];
            for (uint32_t v = tid; v < nvec; v += DS_THREADS) {
                const uint32_t k0 = head + 16u * v, wi = k0 >> 2, bs = (k0 & 3u) * 8u;
                const uint32_t a0 = s_out32[wi], a1 = s_out32[wi + 1], a2 = s_out32[wi + 2], a3 = s_out32[wi + 3], a4 = s_out32[wi + 4];
                uint4 o4;
                o4.x = __funnelshift_r(a0, a1, bs); o4.y = __funnelshift_r(a1, a2, bs);
                o4.z = __funnelshift_r(a2, a3, bs); o4.w = __funnelshift_r(a3, a4, bs);
                *reinterpret_cast<uint4 *>(dst + k0) = o4;
            }
        }
        if (RST) {   // the interval after marker j begins at the output offset of the first byte kept after it
#pragma unroll
            for (int p = 0; p < DS_NP; p++) {
                if (mark[p]) {
                    uint32_t j = (uint32_t)(s_goff >> DS_MK_SHIFT) + (ex[p] >> 16), oo = ex[p] & 0xFFFFu;
                    for (int i = 0; i < 16; i++) {
                        if (mark[p] & (1u << i)) {
                            if (j < bnd_cap) bnd[j] = (uint32_t)(goff + oo); else atomicOr(err, 16u);
                            j++;
                        }
                        if (keep[p] & (1u << i)) oo++;
                    }
                }
            }
        }
        if (ch == c1 - 1 && tid == 0) *avail = goff + tkept;
        if (ch == nchunks - 1) {
            if (tid < 64) dst[tkept + tid] = 0xFF;  // padding the bit reader may peek into
            if (tid == 0) {
                *out_len = goff + tkept;
                if (RST) {
                    const uint32_t nm = (uint32_t)(s_goff >> DS_MK_SHIFT) + (total >> 16);
                    *nmark = nm;
                    if (nm < bnd_cap) bnd[nm] = 0xFFFFFFFFu; else atomicOr(err, 16u);
                }
            }
        }
        __syncthreads();
        for (uint32_t i = tid; i * 16 < tkept + 20; i += DS_THREADS) reinterpret_cast<uint4 *>(s_out32)[i] = make_uint4(0, 0, 0, 0);
    }
}

// ------------------------------------------------------------------------------------------------------
// Huffman decoding of one symbol from the top 16 bits of a window (jdhuff.c jpeg_huff_decode, table-driven)
__device__ __forceinline__ uint32_t huff_sym(const uint16_t *lut, const int32_t *maxcode, const int32_t *valoff,
                                             const uint8_t *vals, uint32_t top16, int &len) {
    const uint32_t e = lut[top16 >> (16 - DEC_LUT_BITS)];
    if (e) {
        len = (int)(e >> 8);
        return e & 0xFFu;
    }
#pragma unroll 1
    for (int l = DEC_LUT_BITS + 1; l <= 16; l++) {
        const int code = (int)(top16 >> (16 - l));
        if (code <= maxcode[l]) {
            len = l;
            return vals[(valoff[l] + code) & 255];
        }
    }
    len = 1;  // invalid code (only reached while unsynchronised): skip one bit and keep going (SURVEY.md App. D)
    return 0x100u;
}

constexpr int SUB_BITS = 1024;                 // subsequence length
constexpr int SUB_WORDS = SUB_BITS / 32;
constexpr int DEC_THREADS = 256;               // subsequences per CTA
constexpr int DEC_FIRST_SKIP = 512;            // bits of every subsequence the first synchronisation pass does not decode
// The chunk's words live at g + (g >> 5): one pad word per subsequence, so threads that stand at the same word of their
// own subsequences hit 32 different banks, and the address is one shift and one add per load.
constexpr int DEC_SMEM_WORDS = SUB_WORDS * (DEC_THREADS + 1) + DEC_THREADS + 1 + 8;   // + one subsequence of lead-in (k_dec_sync)
__device__ __forceinline__ uint32_t dec_widx(uint32_t g) { return g + (g >> 5); }

struct DecShared {
    uint32_t words[DEC_SMEM_WORDS];            // word g of the staged bits (lead-in + chunk + 2 of overflow) at dec_widx(g)
    uint16_t lut[4][1 << DEC_LUT_BITS];
    int32_t maxcode[4][18];
    int32_t valoff[4][17];
    uint8_t vals[4][256];
    uint64_t state[DEC_THREADS + 1];           // [i + 1] = end state of subsequence i; [0] = state entering the chunk
    uint64_t used[DEC_THREADS];                // the start state that produced state[i + 1]
    uint32_t nblk[DEC_THREADS];
    uint16_t list[DEC_THREADS];                // subsequences to decode this round, compacted
    uint32_t wcnt[DEC_THREADS / 32];
};

// state word: bit position << 16 | block-in-MCU << 8 | zig-zag index
__device__ __forceinline__ uint64_t pack_state(uint64_t p, int c, int k) { return (p << 16) | ((uint64_t)c << 8) | (uint64_t)k; }

// codes longer than the LUT covers (rare), or an invalid code (only while unsynchronised): canonical search
template <class SH>
__device__ __noinline__ uint32_t huff_sym_long(const SH &sh, uint32_t t, uint32_t top16) {
#pragma unroll 1
    for (int l = DEC_LUT_BITS + 1; l <= 16; l++) {
        const int code = (int)(top16 >> (16 - l));
        if (code <= sh.maxcode[t][l]) return ((uint32_t)l << 8) | sh.vals[t][(sh.valoff[t][l] + code) & 255];
    }
    return 0xFFFFu;  // invalid: skip one bit and keep going (SURVEY.md App. D)
}

// Restart intervals (jdhuff.c process_restart): bnd[j] = byte offset in the unstuffed stream where interval j + 1
// begins (k_destuff<true>), closed by 0xFFFFFFFF. At such a position the decoder is at the start of an MCU with
// nothing pending; the bits before it that do not hold a whole symbol are the 1-padding of the interval's last byte
// (no code is all ones, so a symbol read from the padding always runs across the boundary). A decoder that is not
// synchronised yet obeys the same two rules, which is what makes every boundary a synchronisation point.
struct RstTrack {
    const uint32_t *bnd;
    uint32_t j, lim;   // next boundary: index, and position in bits relative to the chunk (0xFFFFFFFF: none in reach)
    uint64_t chunk_bit0;
    __device__ __forceinline__ void load() {
        const uint32_t b = bnd[j];
        const uint64_t rel = (uint64_t)b * 8 - chunk_bit0;
        lim = (b == 0xFFFFFFFFu || rel > 0x7FFFFFFFull) ? 0xFFFFFFFFu : (uint32_t)rel;
    }
    __device__ __forceinline__ void init(const uint32_t *b, uint32_t nmark, uint64_t cb0, uint32_t q) {
        bnd = b; chunk_bit0 = cb0;
        const uint64_t pos = cb0 + q;
        uint32_t lo = 0, hi = nmark;   // smallest j with bnd[j] * 8 >= pos (bnd[nmark] is the sentinel)
        while (lo < hi) {
            const uint32_t mid = (lo + hi) >> 1;
            if ((uint64_t)b[mid] * 8 >= pos) hi = mid; else lo = mid + 1;
        }
        j = lo;
        load();
    }
    __device__ __forceinline__ void next() { j++; load(); }
};

// Decodes from `start_state` up to `end_bit` (jdhuff.c decode_mcu, one symbol per iteration). Positions are kept
// relative to the chunk (32-bit); the block state machine (DC / coefficient / ZRL / EOB) is branch-free.
template <bool WRITE, bool RST>
__device__ __forceinline__ uint64_t decode_range(const DecShared &sh, uint64_t chunk_bit0, uint64_t start_state,
                                                 uint64_t end_bit, uint64_t total_bits, int bpm, int hv,
                                                 uint32_t &nblk_out, int16_t *__restrict__ coef, uint32_t blk_base,
                                                 uint32_t nblocks, const uint32_t *__restrict__ bnd, uint32_t nmark) {
    uint32_t q = (uint32_t)((start_state >> 16) - chunk_bit0);
    int c = (int)((start_state >> 8) & 0xFF), k = (int)(start_state & 0xFF);
    uint32_t nblk = 0;
    const uint64_t left = total_bits - chunk_bit0;
    const uint32_t tot = left > 0x7FFFFFFFull ? 0x7FFFFFFFu : (uint32_t)left;          // end of the stream, clamped
    const uint32_t stop = min((uint32_t)(end_bit - chunk_bit0), tot);
    const uint16_t *lut = &sh.lut[0][0];
    RstTrack rt;
    if (RST) rt.init(bnd, nmark, chunk_bit0, q);
    while (q < stop) {
        if (RST && q >= rt.lim) { c = 0; k = 0; rt.next(); }   // an interval begins here
        const uint32_t g = q >> 5, o = q & 31u;
        const uint32_t w0 = sh.words[dec_widx(g)];
        const uint32_t w1 = sh.words[dec_widx(g + 1)];
        const uint32_t win = __funnelshift_l(w1, w0, o);  // 32 bits starting at q
        const bool dc = k == 0;
        const uint32_t t = (c < hv ? 0u : 2u) + (dc ? 0u : 1u);
        uint32_t e = lut[(t << DEC_LUT_BITS) + (win >> (32 - DEC_LUT_BITS))];
        if (e == 0) e = huff_sym_long(sh, t, win >> 16);
        if (e == 0xFFFFu) {                                  // invalid code
            if (RST && q + 16 > rt.lim) { q = rt.lim; c = 0; k = 0; rt.next(); continue; }   // ... in the padding of an interval
            q += 1;
            continue;
        }
        const uint32_t len = e >> 8, s = e & 15u, r = (e >> 4) & 15u;
        if (RST && q + len + s > rt.lim) { q = rt.lim; c = 0; k = 0; rt.next(); continue; }   // padding before a restart marker
        if (q + len + s > tot) { q = tot; break; }         // padding bits at the very end
        int val = 0;
        if (s) {
            const uint32_t v = (win << len) >> (32 - s);
            val = v < (1u << (s - 1)) ? (int)v - (1 << s) + 1 : (int)v;  // jdhuff.c HUFF_EXTEND
        }
        q += len + s;
        // DC: k = 1. Coefficient: stored at k + r, k += r + 1. ZRL: k += 16. EOB: block done. k > 63: block done.
        int knew = s ? k + (int)r + 1 : (r == 15u ? k + 16 : 64);
        if (dc) knew = 1;
        if (WRITE && s) {
            const uint32_t b = blk_base + nblk;
            const int idx = dc ? 0 : k + (int)r;
            if (idx < 64 && b < nblocks) coef[(size_t)b * 64 + idx] = (int16_t)val;
        }
        const bool done = knew > 63;
        k = done ? 0 : knew;
        c += done ? 1 : 0;
        c = c == bpm ? 0 : c;
        nblk += done ? 1u : 0u;
    }
    nblk_out = nblk;
    return pack_state(chunk_bit0 + q, c, k);
}

__device__ __forceinline__ void dec_load_chunk(DecShared &sh, const uint8_t *__restrict__ u, uint64_t nbytes_padded,
                                               size_t w0, int count, const DecTables *__restrict__ tb) {
    const int tid = threadIdx.x;
    const uint32_t *uw = reinterpret_cast<const uint32_t *>(u);
    const size_t nwords = (size_t)(nbytes_padded >> 2);
    for (int i = tid; i < count; i += DEC_THREADS) {
        const size_t gw = w0 + i;
        const uint32_t w = gw < nwords ? uw[gw] : 0xFFFFFFFFu;
        sh.words[dec_widx((uint32_t)i)] = __byte_perm(w, 0, 0x0123);  // big-endian bit order
    }
    for (int i = tid; i < 4 * (1 << DEC_LUT_BITS); i += DEC_THREADS) (&sh.lut[0][0])[i] = (&tb->lut[0][0])[i];
    for (int i = tid; i < 4 * 18; i += DEC_THREADS) (&sh.maxcode[0][0])[i] = (&tb->maxcode[0][0])[i];
    for (int i = tid; i < 4 * 17; i += DEC_THREADS) (&sh.valoff[0][0])[i] = (&tb->valoff[0][0])[i];
    for (int i = tid; i < 4 * 256; i += DEC_THREADS) (&sh.vals[0][0])[i] = (&tb->vals[0][0])[i];
}

// One synchronisation launch: every CTA iterates up to `inner` rounds over its 256 subsequences (states in shared
// memory), then publishes the end states. st_out[i] = state after subsequence i; st_in[i] = the start state that
// produced it. `changed` is raised when a CTA did not converge or its last end state moved.
// From the third round on only a few subsequences still see a new start state: every round first compacts the
// subsequences that need decoding into a list, and the threads take list entries, so the warps stay full.
template <bool RST>
__global__ void __launch_bounds__(DEC_THREADS)
k_dec_sync(const uint8_t *__restrict__ u, const uint64_t *__restrict__ u_len, const DecTables *__restrict__ tb,
           uint64_t *__restrict__ st_in, uint64_t *__restrict__ st_out, uint32_t *__restrict__ nblk, int bpm, int hv,
           int inner, int mode, uint8_t *__restrict__ done, uint32_t *__restrict__ changed,
           const uint32_t *__restrict__ bnd, const uint32_t *__restrict__ nmark_p, const uint32_t *skip_if_zero) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    DecShared &sh = *reinterpret_cast<DecShared *>(smem_raw);
    if (skip_if_zero && *skip_if_zero == 0u) return;   // the previous launch of the schedule found a fixed point: nothing can move
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const size_t cta = blockIdx.x;
    const uint64_t chunk_bit0 = (uint64_t)cta * SUB_BITS * DEC_THREADS;
    // mode 0: the whole stream is there (*u_len = its length); a chunk whose first pass has not run yet runs it now.
    // mode 1 (stream still arriving, *u_len = bytes de-stuffed so far): only the first pass, only for chunks whose
    //         bytes (and the words the bit reader may peek into) are complete; everything else returns.
    const bool first_launch = done[cta] == 0;
    uint64_t nbytes = *u_len;
    if (mode == 1) {
        if (!first_launch) return;
        if ((chunk_bit0 >> 3) + (uint64_t)(SUB_BITS / 8) * DEC_THREADS + 64 > nbytes) return;
        nbytes = ~0ull >> 8;   // no end of stream inside this chunk
    }
    const uint64_t total_bits = nbytes * 8;
    if (chunk_bit0 >= total_bits) return;
    const uint32_t nmark = RST ? *nmark_p : 0u;
    const size_t i = cta * DEC_THREADS + tid;
    const uint64_t my_bit0_pre = chunk_bit0 + (uint64_t)tid * SUB_BITS;
    // A later launch has work only where a start state differs from the one the subsequence was last decoded from:
    // nothing of the chunk is loaded before that is known (after the first launch most chunks have nothing left to do).
    if (!first_launch) {
        const bool need0 = my_bit0_pre < total_bits && (i == 0 ? pack_state(0, 0, 0) : st_out[i - 1]) != st_in[i];
        if (!__syncthreads_or(need0)) return;
    }
    // The staged bits begin one subsequence before the chunk (lead-in): in the first round thread 0 decodes the second
    // half of it from a guess, which almost always ends in step, so the chunk's own first subsequence starts from the
    // right state in this very launch instead of waiting for the previous chunk's result in the next one.
    const int lead = cta ? 1 : 0;
    const uint64_t base_bit0 = chunk_bit0 - (uint64_t)lead * SUB_BITS;
    dec_load_chunk(sh, u, mode == 1 ? *u_len & ~(uint64_t)3 : (nbytes + 64) & ~(uint64_t)3, (size_t)(base_bit0 >> 5),
                   SUB_WORDS * (DEC_THREADS + lead) + 2, tb);
    const uint64_t my_bit0 = chunk_bit0 + (uint64_t)tid * SUB_BITS;
    const uint64_t my_end = my_bit0 + SUB_BITS;
    const bool live = my_bit0 < total_bits;
    // incoming state of the CTA's first subsequence; first launch: found in round 0 from the lead-in (until then the
    // guess "a block starts exactly at my first bit")
    if (tid == 0) sh.state[0] = cta == 0 ? pack_state(0, 0, 0) : (first_launch ? pack_state(chunk_bit0, 0, 0) : st_out[i - 1]);
    sh.used[tid] = first_launch ? ~0ull : st_in[i];
    const uint64_t before = first_launch ? pack_state(my_end, 0, 0) : st_out[i];
    sh.nblk[tid] = first_launch ? 0 : nblk[i];
    sh.state[tid + 1] = before;
    __syncthreads();
    int any = 1;
    for (int round = 0; round < inner && any; round++) {
        // ---- who needs decoding: start state differs from the one used last time
        const bool need = live && sh.state[tid] != sh.used[tid];
        const unsigned bal = __ballot_sync(0xffffffffu, need);
        if (lane == 0) sh.wcnt[wid] = __popc(bal);
        __syncthreads();
        uint32_t wbase = 0, total = 0;
#pragma unroll
        for (int w = 0; w < DEC_THREADS / 32; w++) { const uint32_t x = sh.wcnt[w]; if (w < wid) wbase += x; total += x; }
        if (need) sh.list[wbase + __popc(bal & ((1u << lane) - 1u))] = (uint16_t)tid;
        __syncthreads();
        // ---- decode the listed subsequences (their start states are read before anybody writes an end state)
        int ch = 0;
        uint64_t outst = 0, in = 0;
        uint32_t nb = 0;
        int t = -1;
        bool leadin = false;
        if ((uint32_t)tid < total) {
            t = sh.list[tid];
            in = sh.state[t];
            uint64_t t_end = chunk_bit0 + (uint64_t)(t + 1) * SUB_BITS;
            uint64_t from = in;
            // The very first pass only looks for a synchronisation point: every start state is a guess and the block
            // counts are thrown away (the next round decodes again from the real states), so it decodes the second half
            // of the subsequence only -- a decoder is in step after one or two hundred bits on ordinary streams.
            // Thread 0 of a chunk other than the first spends that pass on the lead-in: its end is the chunk's start state.
            if (first_launch && round == 0 && !(cta == 0 && t == 0)) {
                leadin = t == 0;
                from = pack_state(chunk_bit0 + (uint64_t)t * SUB_BITS + DEC_FIRST_SKIP - (leadin ? (uint64_t)SUB_BITS : 0), 0, 0);
                if (leadin) t_end = chunk_bit0;
                in = ~0ull;
            }
            outst = decode_range<false, RST>(sh, base_bit0, from, t_end, total_bits, bpm, hv, nb, nullptr, 0, 0, bnd, nmark);
        }
        __syncthreads();
        if (t >= 0) {
            if (leadin) {   // the chunk's start state; subsequence 0 itself is decoded from it in the next round
                sh.state[0] = outst;
                ch = 1;
            } else {
                ch = outst != sh.state[t + 1];
                sh.state[t + 1] = outst;
                sh.used[t] = in;
                sh.nblk[t] = nb;
            }
        }
        any = __syncthreads_or(ch);
    }
    const uint64_t mine = sh.state[tid + 1], used = sh.used[tid];
    if (live) {
        st_in[i] = used;
        st_out[i] = mine;
        nblk[i] = sh.nblk[tid];
    }
    if (tid == 0) done[cta] = 1;
    // not converged inside the CTA, or the state handed to the next CTA moved
    const bool last_live = tid == DEC_THREADS - 1 || my_end >= total_bits;
    if (any || (live && last_live && mine != before) || (live && sh.state[tid] != used)) atomicOr(changed, 1u);
}

// ------------------------------------------------------------------------------------------------------
// k_dec_sync_long: the synchronisation for streams with LONG synchronisation distances (q100: blocks rarely end with
// EOB, so a decoder that starts out of phase stays out of phase for many kilobits) and for the checked retry. One
// thread decodes a GROUP of `DEC_GROUP` (8 ... 64, chosen by the host) consecutive subsequences in one go (a streaming bit reader on the unstuffed
// bytes in global memory), recording the state at every 1024-bit boundary on the way, so k_scan_u32 / k_dec_write see
// the same per-subsequence arrays as after k_dec_sync -- but a launch costs one pass over the stream and carries a
// correction DEC_GROUP subsequences further, where k_dec_sync re-decodes every subsequence once per subsequence of
// distance. A group whose start state did not change since it was last decoded is skipped.
constexpr int DEC_LONG_THREADS = 128;
struct DecTabShared {
    uint16_t lut[4][1 << DEC_LUT_BITS];
    int32_t maxcode[4][18];
    int32_t valoff[4][17];
    uint8_t vals[4][256];
};

template <bool RST>
__global__ void __launch_bounds__(DEC_LONG_THREADS)
k_dec_sync_long(const uint8_t *__restrict__ u, const uint64_t *__restrict__ u_len, const DecTables *__restrict__ tb,
                uint64_t *__restrict__ st_in, uint64_t *__restrict__ st_out, uint32_t *__restrict__ nblk, int bpm, int hv,
                int first, int DEC_GROUP, uint32_t *__restrict__ changed, const uint32_t *__restrict__ bnd,
                const uint32_t *__restrict__ nmark_p) {
    __shared__ DecTabShared sh;
    const int tid = threadIdx.x;
    for (int i = tid; i < 4 * (1 << DEC_LUT_BITS); i += DEC_LONG_THREADS) (&sh.lut[0][0])[i] = (&tb->lut[0][0])[i];
    for (int i = tid; i < 4 * 18; i += DEC_LONG_THREADS) (&sh.maxcode[0][0])[i] = (&tb->maxcode[0][0])[i];
    for (int i = tid; i < 4 * 17; i += DEC_LONG_THREADS) (&sh.valoff[0][0])[i] = (&tb->valoff[0][0])[i];
    for (int i = tid; i < 4 * 256; i += DEC_LONG_THREADS) (&sh.vals[0][0])[i] = (&tb->vals[0][0])[i];
    __syncthreads();
    const uint64_t nbytes = *u_len;
    const uint64_t total_bits = nbytes * 8;
    const size_t grp = (size_t)blockIdx.x * DEC_LONG_THREADS + tid;
    const size_t sub0 = grp * DEC_GROUP;
    const uint64_t bit0 = (uint64_t)sub0 * SUB_BITS;
    if (bit0 >= total_bits) return;
    // start state: the stream's start, the guess "a block starts exactly at my first bit" (first launch), or what the
    // previous group reached in the previous launch
    const uint64_t in = grp == 0 ? pack_state(0, 0, 0) : (first ? pack_state(bit0, 0, 0) : st_out[sub0 - 1]);
    if (!first && in == st_in[sub0]) return;   // nothing new for this group
    st_in[sub0] = in;
    uint64_t q = in >> 16;                      // absolute bit position
    int c = (int)((in >> 8) & 0xFF), k = (int)(in & 0xFF);
    // streaming bit reader: acc holds the next `nav` bits left-aligned; words come from a four-word register queue that
    // is refilled with 16-byte loads issued one vector ahead (a thread walks alone through its kilobytes: the load
    // latency must not sit on the symbol chain)
    const uint4 *u4 = reinterpret_cast<const uint4 *>(u);
    uint64_t acc = 0;
    int nav = 0, qn = 0;           // qn: words left in the queue
    uint32_t w0 = 0, w1 = 0, w2 = 0, w3 = 0;
    uint4 ahead = make_uint4(0, 0, 0, 0);
    size_t vidx = 0;               // index of the vector in `ahead`
    auto next_word = [&]() -> uint32_t {
        if (qn == 0) {
            w0 = ahead.x; w1 = ahead.y; w2 = ahead.z; w3 = ahead.w;
            qn = 4;
            vidx++;
            ahead = u4[vidx];
        }
        const uint32_t w = w0;
        w0 = w1; w1 = w2; w2 = w3;
        qn--;
        return __byte_perm(w, 0, 0x0123);
    };
    auto seek = [&](uint64_t pos) {
        const size_t widx = (size_t)(pos >> 5);
        vidx = widx >> 2;
        const uint4 cur = u4[vidx];
        w0 = cur.x; w1 = cur.y; w2 = cur.z; w3 = cur.w;
        qn = 4;
        vidx++;
        ahead = u4[vidx];
        for (int i = 0; i < (int)(widx & 3); i++) { w0 = w1; w1 = w2; w2 = w3; qn--; }
        const uint32_t a = next_word(), b = next_word();
        acc = (((uint64_t)a << 32) | b) << (pos & 31u);
        nav = 64 - (int)(pos & 31u);
    };
    seek(q);
    uint64_t lim = ~0ull;   // next restart boundary (absolute bits)
    uint32_t bj = 0;
    if (RST) {
        const uint32_t nm = *nmark_p;
        uint32_t lo = 0, hi = nm;
        while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if ((uint64_t)bnd[mid] * 8 >= q) hi = mid; else lo = mid + 1; }
        bj = lo;
        lim = bnd[bj] == 0xFFFFFFFFu ? ~0ull : (uint64_t)bnd[bj] * 8;
    }
    const uint16_t *lut = &sh.lut[0][0];
    uint32_t nb = 0;
    int j = 0;                                  // subsequence of the group that is being decoded
    uint64_t sub_end = min(bit0 + SUB_BITS, total_bits);
    bool moved = false;
    // the state at the first symbol boundary at or past a subsequence's end is that subsequence's end state
    auto record = [&]() {
        while (j < DEC_GROUP && q >= sub_end) {
            const size_t si = sub0 + j;
            const uint64_t stt = pack_state(q, c, k);
            if (j == DEC_GROUP - 1 || sub_end >= total_bits) moved = moved || first || st_out[si] != stt;
            st_out[si] = stt;
            nblk[si] = nb;
            nb = 0;
            j++;
            if (sub_end >= total_bits) { j = DEC_GROUP; break; }
            sub_end = min(sub_end + SUB_BITS, total_bits);
            if (j < DEC_GROUP) st_in[sub0 + j] = stt;
        }
    };
    record();
    while (j < DEC_GROUP) {
        if (RST && q >= lim) { c = 0; k = 0; bj++; lim = bnd[bj] == 0xFFFFFFFFu ? ~0ull : (uint64_t)bnd[bj] * 8; }
        if (nav <= 32) {
            acc |= (uint64_t)next_word() << (32 - nav);
            nav += 32;
        }
        const uint32_t win = (uint32_t)(acc >> 32);
        const bool dc = k == 0;
        const uint32_t t = (c < hv ? 0u : 2u) + (dc ? 0u : 1u);
        uint32_t e = lut[(t << DEC_LUT_BITS) + (win >> (32 - DEC_LUT_BITS))];
        if (e == 0) e = huff_sym_long(sh, t, win >> 16);
        uint32_t adv;
        if (e == 0xFFFFu) {
            if (RST && q + 16 > lim) { q = lim; c = 0; k = 0; bj++; lim = bnd[bj] == 0xFFFFFFFFu ? ~0ull : (uint64_t)bnd[bj] * 8; seek(q); record(); continue; }
            adv = 1;                             // invalid code (only while unsynchronised): skip one bit
        } else {
            const uint32_t len = e >> 8, sz = e & 15u, r = (e >> 4) & 15u;
            adv = len + sz;
            if (RST && q + adv > lim) { q = lim; c = 0; k = 0; bj++; lim = bnd[bj] == 0xFFFFFFFFu ? ~0ull : (uint64_t)bnd[bj] * 8; seek(q); record(); continue; }
            if (q + adv > total_bits) { q = total_bits; record(); break; }   // padding bits at the very end
            int knew = sz ? k + (int)r + 1 : (r == 15u ? k + 16 : 64);
            if (dc) knew = 1;
            const bool done = knew > 63;
            k = done ? 0 : knew;
            c = done ? (c + 1 == bpm ? 0 : c + 1) : c;
            nb += done ? 1u : 0u;
        }
        q += adv;
        acc <<= adv;
        nav -= (int)adv;
        if (q >= sub_end) record();
    }
    if (moved) atomicOr(changed, 1u);
}

// Final pass: decode every subsequence from its synchronised start state and write whole coefficient blocks
// (zig-zag order, DC still differential). A block belongs to the thread in whose subsequence it STARTS: that thread
// keeps decoding past its last bit until the block is complete (a block is at most 1665 bits: two subsequences of
// lookahead are staged), and skips the tail of the block that was running when its subsequence began. The owner
// collects the block's coefficients in a 128-byte cell of shared memory; the warp runs in lock step, one symbol per
// lane and iteration, and after every iteration the lanes that completed a block have it written out by the whole
// warp: one coalesced 128-byte store per block, zeros included -- no memset of the array, no scattered 2-byte stores.
struct DecWriteShared {
    uint32_t words[SUB_WORDS * (DEC_THREADS + 2) + DEC_THREADS + 2 + 8];   // 256 subsequences + 2 of lookahead, word g at dec_widx(g)
    uint16_t lut[4][1 << DEC_LUT_BITS];
    int32_t maxcode[4][18];
    int32_t valoff[4][17];
    uint8_t vals[4][256];
    uint32_t blk[DEC_THREADS][32];                   // word w of thread t's block at [t][w ^ (t & 31)]
};

template <bool RST>
__global__ void __launch_bounds__(DEC_THREADS)
k_dec_write(const uint8_t *__restrict__ u, const uint64_t *__restrict__ u_len, const DecTables *__restrict__ tb,
            const uint64_t *__restrict__ st_out, const uint32_t *__restrict__ blk_start, int bpm, int hv,
            int16_t *__restrict__ coef, int16_t *__restrict__ dcarr, uint32_t nblocks, uint32_t *__restrict__ err,
            const uint32_t *__restrict__ bnd, const uint32_t *__restrict__ nmark_p) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    DecWriteShared &sh = *reinterpret_cast<DecWriteShared *>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31;
    const uint64_t nbytes = *u_len;
    const uint64_t total_bits = nbytes * 8;
    const size_t cta = blockIdx.x;
    const uint64_t chunk_bit0 = (uint64_t)cta * SUB_BITS * DEC_THREADS;
    if (chunk_bit0 >= total_bits) return;
    {   // the chunk's words + two subsequences of lookahead, tables, empty block cells
        const uint32_t *uw = reinterpret_cast<const uint32_t *>(u);
        const size_t w0 = cta * (size_t)(SUB_WORDS * DEC_THREADS);
        const size_t nwords = (size_t)(((nbytes + 64) & ~(uint64_t)3) >> 2);
        for (int i = tid; i < SUB_WORDS * (DEC_THREADS + 2); i += DEC_THREADS) {
            const size_t gw = w0 + i;
            const uint32_t w = gw < nwords ? uw[gw] : 0xFFFFFFFFu;
            sh.words[dec_widx((uint32_t)i)] = __byte_perm(w, 0, 0x0123);  // big-endian bit order
        }
        for (int i = tid; i < 4 * (1 << DEC_LUT_BITS); i += DEC_THREADS) (&sh.lut[0][0])[i] = (&tb->lut[0][0])[i];
        for (int i = tid; i < 4 * 18; i += DEC_THREADS) (&sh.maxcode[0][0])[i] = (&tb->maxcode[0][0])[i];
        for (int i = tid; i < 4 * 17; i += DEC_THREADS) (&sh.valoff[0][0])[i] = (&tb->valoff[0][0])[i];
        for (int i = tid; i < 4 * 256; i += DEC_THREADS) (&sh.vals[0][0])[i] = (&tb->vals[0][0])[i];
#pragma unroll
        for (int w = 0; w < 32; w++) sh.blk[tid][w ^ lane] = 0;
    }
    __syncthreads();
    const size_t i = cta * DEC_THREADS + tid;
    const uint64_t my_bit0 = chunk_bit0 + (uint64_t)tid * SUB_BITS;
    const bool live = my_bit0 < total_bits;
    const uint64_t in = (!live || i == 0) ? pack_state(live ? 0 : my_bit0, 0, 0) : st_out[i - 1];
    uint32_t q = (uint32_t)((in >> 16) - chunk_bit0);
    int c = (int)((in >> 8) & 0xFF), k = (int)(in & 0xFF);
    const uint64_t left = total_bits - chunk_bit0;
    const uint32_t tot = left > 0x7FFFFFFFull ? 0x7FFFFFFFu : (uint32_t)left;
    const uint32_t stop = min((uint32_t)(tid + 1) * SUB_BITS, tot);
    uint32_t b_cur = live ? blk_start[i] : 0;   // index of the block that is running (or starts) at q
    bool owning = k == 0;                        // a block that starts here is mine; a running one is my predecessor's
    bool active = live && !(k == 0 && q >= stop);
    bool crossed = q >= stop;                    // the state at the first symbol boundary at or past `stop` must be st_out[i]
    uint64_t end_state = in;
    const uint16_t *lut = &sh.lut[0][0];
    uint32_t *cell = sh.blk[tid];
    RstTrack rt;
    if (RST) rt.init(bnd, *nmark_p, chunk_bit0, q);
    while (__any_sync(0xffffffffu, active)) {
        bool flush = false;
        if (active) {
            if (RST && q >= rt.lim) { c = 0; k = 0; rt.next(); }   // an interval begins here (states are synchronised: nothing pending)
            const uint32_t g = q >> 5, o = q & 31u;
            const uint32_t w0 = sh.words[dec_widx(g)];
            const uint32_t w1 = sh.words[dec_widx(g + 1)];
            const uint32_t win = __funnelshift_l(w1, w0, o);
            const bool dc = k == 0;
            const uint32_t t = (c < hv ? 0u : 2u) + (dc ? 0u : 1u);
            uint32_t e = lut[(t << DEC_LUT_BITS) + (win >> (32 - DEC_LUT_BITS))];
            if (e == 0) e = huff_sym_long(sh, t, win >> 16);
            const uint32_t len = e >> 8, s = e & 15u, r = (e >> 4) & 15u;
            if (RST && ((e == 0xFFFFu && q + 16 > rt.lim) || (e != 0xFFFFu && q + len + s > rt.lim))) {
                // the 1-padding before a restart marker: the next interval (and block) begins at the boundary
                q = rt.lim; c = 0; k = 0;
                rt.next();
                owning = true;
                if (q >= stop) active = false;   // blocks that start at or past my last bit are not mine
            } else if (e == 0xFFFFu || q + len + s > tot) {   // cannot happen on synchronised states except in the final padding
                q = tot;
                active = false;
            } else {
                int val = 0;
                if (s) {
                    const uint32_t v = (win << len) >> (32 - s);
                    val = v < (1u << (s - 1)) ? (int)v - (1 << s) + 1 : (int)v;  // jdhuff.c HUFF_EXTEND
                }
                q += len + s;
                int knew = s ? k + (int)r + 1 : (r == 15u ? k + 16 : 64);
                if (dc) knew = 1;
                if (owning && s) {
                    const int idx = dc ? 0 : k + (int)r;
                    if (idx < 64) reinterpret_cast<int16_t *>(&cell[(idx >> 1) ^ lane])[idx & 1] = (int16_t)val;
                }
                // a block ends about once in twenty symbols, i.e. in some lane of the warp in most iterations: no branch here
                const bool done = knew > 63;
                k = done ? 0 : knew;
                c += done ? 1 : 0;
                c = c == bpm ? 0 : c;
                flush = done && owning;
                b_cur += (done && !owning) ? 1u : 0u;          // my predecessor's block is over; the next one is mine
                owning = owning || done;
                active = !(done && q >= stop);                 // blocks that start at or past my last bit are not mine
            }
            if (!crossed && q >= stop) { crossed = true; end_state = pack_state(chunk_bit0 + q, c, k); }
        }
        // ---- completed blocks: the whole warp writes each one (128 bytes, coalesced) and clears its cell
        __syncwarp();
        unsigned fl = __ballot_sync(0xffffffffu, flush);
        while (fl) {
            const int L = __ffs(fl) - 1;
            fl &= fl - 1;
            const uint32_t b = __shfl_sync(0xffffffffu, b_cur, L);
            uint32_t *src = sh.blk[(tid & ~31) + L];
            const uint32_t w = src[lane ^ L];
            src[lane ^ L] = 0;
            if (b < nblocks) {
                reinterpret_cast<uint32_t *>(coef)[(size_t)b * 32 + lane] = w;
                if (lane == 0) dcarr[b] = (int16_t)(w & 0xFFFFu);   // the DC differences also go to a compact array (k_dc_scan)
            }
        }
        if (flush) b_cur++;
        __syncwarp();
    }
    if (live && (!crossed || end_state != st_out[i])) atomicOr(err, 4u);  // the states were not a fixed point
}

// ------------------------------------------------------------------------------------------------------
// Generic exclusive scan of uint32 (chunked, look-back). out[n] receives the total.
__global__ void __launch_bounds__(256)
k_scan_u32(const uint32_t *__restrict__ in, uint32_t *__restrict__ out, size_t n, uint64_t *__restrict__ desc,
           uint32_t *__restrict__ ticket, uint32_t *__restrict__ err) {
    constexpr int ITEMS = 8, CH = 256 * ITEMS;
    __shared__ int s_chunk;
    __shared__ uint32_t s_warp[8];
    __shared__ uint64_t s_goff;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int nchunks = (int)((n + CH - 1) / CH);
    for (;;) {
        if (tid == 0) s_chunk = (int)atomicAdd(ticket, 1u);
        __syncthreads();
        const int ch = s_chunk;
        if (ch >= nchunks) break;
        const size_t base = (size_t)ch * CH + (size_t)tid * ITEMS;
        uint32_t v[ITEMS], sum = 0;
#pragma unroll
        for (int j = 0; j < ITEMS; j++) { v[j] = base + j < n ? in[base + j] : 0; sum += v[j]; }
        uint32_t inc = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += y;
        }
        if (lane == 31) s_warp[wid] = inc;
        __syncthreads();
        uint32_t wbase = 0, total = 0;
#pragma unroll
        for (int j = 0; j < 8; j++) { const uint32_t x = s_warp[j]; if (j < wid) wbase += x; total += x; }
        if (wid == 0) {
            const uint64_t pre = lookback_exclusive(desc, ch, total, err);
            if (lane == 0) s_goff = pre;
        }
        __syncthreads();
        uint32_t run = (uint32_t)s_goff + wbase + inc - sum;
#pragma unroll
        for (int j = 0; j < ITEMS; j++) { if (base + j < n) out[base + j] = run; run += v[j]; }
        if (ch == nchunks - 1 && tid == 255) out[n] = (uint32_t)s_goff + total;
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------------
// DC un-differencing: inclusive prefix sum of the DC differences of one component over its blocks in scan order
// (jdhuff.c decode_mcu: s += last_dc_val), on the compact array of DCs (one int16 per block) that k_dec_write fills;
// k_idct takes the DC from there. blockIdx.y = component; chunked look-back per component.
__global__ void __launch_bounds__(256)
k_dc_scan(int16_t *__restrict__ coef, int bpm, int hv, size_t nmcu, uint64_t *__restrict__ desc_all,
          uint32_t *__restrict__ ticket_all, size_t desc_stride, uint32_t *__restrict__ err) {
    constexpr int ITEMS = 16, CH = 256 * ITEMS;   // 4096 blocks per look-back unit: few, long chunks keep the walk short
    __shared__ int s_chunk;
    __shared__ int s_warp[8];
    __shared__ uint64_t s_goff;
    const int comp = blockIdx.y;
    uint64_t *desc = desc_all + (size_t)comp * desc_stride;
    uint32_t *ticket = ticket_all + comp;
    const int per = comp == 0 ? hv : 1;
    const size_t n = nmcu * per;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int nchunks = (int)((n + CH - 1) / CH);
    auto index_of = [&](size_t e) -> size_t {   // block index (= index into the compact DC array) of element e of this component
        const size_t m = comp == 0 ? e / hv : e;
        const int sub = comp == 0 ? (int)(e - m * hv) : hv + comp - 1;
        return m * bpm + sub;
    };
    for (;;) {
        if (tid == 0) s_chunk = (int)atomicAdd(ticket, 1u);
        __syncthreads();
        const int ch = s_chunk;
        if (ch >= nchunks) break;
        const size_t base = (size_t)ch * CH + (size_t)tid * ITEMS;
        int v[ITEMS], sum = 0;
#pragma unroll
        for (int j = 0; j < ITEMS; j++) {
            const size_t e = base + j;
            v[j] = e < n ? (int)coef[index_of(e)] : 0;
            sum += v[j];
        }
        int inc = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += y;
        }
        if (lane == 31) s_warp[wid] = inc;
        __syncthreads();
        int wbase = 0, total = 0;
#pragma unroll
        for (int j = 0; j < 8; j++) { const int x = s_warp[j]; if (j < wid) wbase += x; total += x; }
        if (wid == 0) {
            const uint64_t pre = lookback_exclusive(desc, ch, (uint64_t)(int64_t)total & LB_MASK, err);
            if (lane == 0) s_goff = pre;
        }
        __syncthreads();
        int run = (int)(uint32_t)s_goff + wbase + inc - sum;  // low 32 bits of the modular sum are exact
#pragma unroll
        for (int j = 0; j < ITEMS; j++) {
            run += v[j];
            if (base + j < n) coef[index_of(base + j)] = (int16_t)run;
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------------
// k_idct: de-quantise + jidctint.c jpeg_idct_islow, one thread per block, samples to per-component planes.
// Persistent CTAs (two per SM: 128 registers per thread) walk tiles of 256 blocks; the tile's 32 KB of coefficients
// arrive by cp.async (16 bytes per request, written straight to their bank-swizzled place) into one of two shared
// buffers while the previous tile is transformed, so the load latency that used to sit in front of every tile's
// arithmetic is hidden. The de-quantisation table is kept as 32-bit words in zig-zag order (one 16-byte load per four
// coefficients); samples are clamped with the fused add-min/max and packed with byte permutes.
constexpr int IDCT_TILE = 256;
constexpr int IDCT_SMEM = 2 * IDCT_TILE * 8 * 16;

__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// GRAY: only the luma blocks are transformed and their samples go straight to the caller's 8-bit image (py, pitch
// out_step), cut at the image's right and bottom edges: no Y plane in between (it would cost two more passes over W * H
// bytes) and no colour kernel behind it.
template <bool GRAY>
__global__ void __launch_bounds__(256, 2)
k_idct(const int16_t *__restrict__ coef, const int16_t *__restrict__ dcarr, Geom g, const DecTables *__restrict__ tb,
       uint8_t *__restrict__ py, uint8_t *__restrict__ pcb, uint8_t *__restrict__ pcr, int rst_mcus, size_t out_step) {
    extern __shared__ __align__(16) uint4 s_c[];   // [2][IDCT_TILE * 8], chunk c of block b at b * 8 + (c ^ (b & 7))
    __shared__ __align__(16) int s_q[2][64];       // zig-zag order
    const int tid = threadIdx.x;
    const int ntile = (g.nblocks + IDCT_TILE - 1) / IDCT_TILE;
    const uint4 *coef4 = reinterpret_cast<const uint4 *>(coef);
    auto issue = [&](int tile, int buf) {
        const int b0 = tile * IDCT_TILE, nb = min(IDCT_TILE, g.nblocks - b0);
        uint4 *dstb = s_c + buf * (IDCT_TILE * 8);
        for (int i = tid; i < nb * 8; i += 256) {
            const int b = i >> 3, c = i & 7;
            cp_async16(dstb + b * 8 + (c ^ (b & 7)), coef4 + (size_t)b0 * 8 + i);
        }
        cp_async_commit();
    };
    int t = blockIdx.x;
    if (t < ntile) issue(t, 0);
    if (tid < 128) s_q[tid >> 6][tid & 63] = (int)tb->q[tid >> 6][zigzag_nat_rt(tid & 63)];
    const int hv = GRAY ? g.hs * g.vs : g.bpm - 2;   // luma blocks per MCU (a colour file on a gray context keeps its chroma)
    for (int k = 0; t < ntile; t += gridDim.x, k++) {
        const int tn = t + gridDim.x;
        if (tn < ntile) { issue(tn, (k + 1) & 1); cp_async_wait<1>(); }
        else cp_async_wait<0>();
        __syncthreads();   // tile t has landed (every thread waited for its own requests)
        const int b0 = t * IDCT_TILE, nb = min(IDCT_TILE, g.nblocks - b0);
        if (tid < nb && (!GRAY || (b0 + tid) % g.bpm < hv)) {
            const uint4 *sc = s_c + (k & 1) * (IDCT_TILE * 8);
            const int b = b0 + tid;
            const int m = b / g.bpm, bn = b - m * g.bpm;
            const int my = m / g.mcux, mx = m - my * g.mcux;
            const bool isY = bn < hv;
            const int4 *q4 = reinterpret_cast<const int4 *>(s_q[isY ? 0 : 1]);
            int v[64];
            int c0raw = 0;
#pragma unroll
            for (int ch = 0; ch < 8; ch++) {
                const uint4 w = sc[tid * 8 + (ch ^ (tid & 7))];
                const uint32_t ww[4] = {w.x, w.y, w.z, w.w};
                const int4 qa = q4[2 * ch], qb = q4[2 * ch + 1];
                const int qq[8] = {qa.x, qa.y, qa.z, qa.w, qb.x, qb.y, qb.z, qb.w};
                if (ch == 0) c0raw = (int)(int16_t)(w.x & 0xFFFFu);
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    const int n = zigzag_nat(ch * 8 + j);
                    const int cv = (j & 1) ? ((int)ww[j >> 1] >> 16) : (int)(int16_t)(ww[j >> 1] & 0xFFFFu);
                    v[n] = cv * qq[j];
                }
            }
            // the un-differenced DC (the coefficient array holds the difference): k_dc_scan's running sum, taken from the
            // start of the block's restart interval (predictors return to 0 there; 16-bit modular differences are exact)
            // (dcarr == NULL: the blocks come from the encoder and hold the quantised DC itself -- b2j_reconstruct_*)
            int dcv = dcarr ? (int)dcarr[b] : c0raw;
            if (dcarr && rst_mcus > 0 && m >= rst_mcus) {
                const int pm = (m / rst_mcus) * rst_mcus - 1;   // last MCU of the previous interval
                dcv = (int16_t)(dcv - (int)dcarr[pm * g.bpm + (isY ? hv - 1 : bn)]);
            }
            v[0] = dcv * s_q[isY ? 0 : 1][0];
#pragma unroll
            for (int c = 0; c < 8; c++) idct8<11>(v[c], v[8 + c], v[16 + c], v[24 + c], v[32 + c], v[40 + c], v[48 + c], v[56 + c]);
            uint8_t *dst;
            size_t stride;
            int gx0 = 0, nrow = 8;   // GRAY: the block's first column and its rows inside the image
            if (GRAY) {
                const int by = bn / g.hs, bx = bn - by * g.hs;
                const int gy0 = (my * g.vs + by) * 8;
                gx0 = (mx * g.hs + bx) * 8;
                nrow = min(8, g.H - gy0);
                stride = out_step;
                dst = py + (size_t)gy0 * stride + (size_t)gx0;
            } else if (isY) {
                const int by = bn / g.hs, bx = bn - by * g.hs;
                stride = (size_t)g.mcux * 8 * g.hs;
                dst = py + ((size_t)(my * g.vs + by) * 8) * stride + (size_t)(mx * g.hs + bx) * 8;
            } else {
                stride = (size_t)g.mcux * 8;
                dst = (bn == hv ? pcb : pcr) + ((size_t)my * 8) * stride + (size_t)mx * 8;
            }
#pragma unroll
            for (int r = 0; r < 8; r++) {
                idct8<18>(v[r * 8], v[r * 8 + 1], v[r * 8 + 2], v[r * 8 + 3], v[r * 8 + 4], v[r * 8 + 5], v[r * 8 + 6], v[r * 8 + 7]);
                uint32_t x[8];
#pragma unroll
                for (int c = 0; c < 8; c++) x[c] = (uint32_t)min(255, max(0, v[r * 8 + c] + 128));
                const uint32_t lo = __byte_perm(__byte_perm(x[0], x[1], 0x0040), __byte_perm(x[2], x[3], 0x0040), 0x5410);
                const uint32_t hi = __byte_perm(__byte_perm(x[4], x[5], 0x0040), __byte_perm(x[6], x[7], 0x0040), 0x5410);
                if (!GRAY) {
                    *reinterpret_cast<uint2 *>(dst + r * stride) = make_uint2(lo, hi);
                } else if (r < nrow) {
                    uint8_t *d = dst + r * stride;
                    if (gx0 + 8 <= g.W && ((reinterpret_cast<uintptr_t>(d) & 7) == 0)) *reinterpret_cast<uint2 *>(d) = make_uint2(lo, hi);
                    else for (int c = 0; c < min(8, g.W - gx0); c++) d[c] = (uint8_t)x[c];
                }
            }
        }
        __syncthreads();   // buffer k & 1 is free for the tile after next
    }
}

// ------------------------------------------------------------------------------------------------------
// k_upcolor: jdsample.c fancy upsampling (h2v1 / h2v2 / h1v2 triangle filters, h4v1 replication) on the TRUE
// downsampled size + jdcolor.c YCbCr->RGB, 8 pixels per thread, stored interleaved B,G,R (cv::Mat CV_8UC3).
template <int HS, int VS>
__device__ __forceinline__ int chroma_at(const uint8_t *__restrict__ p, size_t stride, int dw, int rlo, int rhi, int x, int y) {
    if (HS == 1 && VS == 1) return p[(size_t)y * stride + x];
    if (HS == 4) return p[(size_t)y * stride + (x >> 2)];
    if (HS == 2 && VS == 1) {
        const uint8_t *row = p + (size_t)y * stride;
        const int i = x >> 1;
        if (dw <= 2) return row[i];
        if (x & 1) return i < dw - 1 ? (3 * row[i] + row[i + 1] + 2) >> 2 : row[dw - 1];
        return i > 0 ? (3 * row[i] + row[i - 1] + 1) >> 2 : row[0];
    }
    if (HS == 1 && VS == 2) {
        const int r = y >> 1;
        const int rn = (y & 1) ? min(r + 1, rhi) : max(r - 1, rlo);
        return (3 * p[(size_t)r * stride + x] + p[(size_t)rn * stride + x] + ((y & 1) ? 2 : 1)) >> 2;
    }
    // h2v2
    const int r = y >> 1, i = x >> 1;
    if (dw <= 2) return p[(size_t)r * stride + i];
    const int rn = (y & 1) ? min(r + 1, rhi) : max(r - 1, rlo);
    const uint8_t *r0 = p + (size_t)r * stride, *r1 = p + (size_t)rn * stride;
    const int s = 3 * r0[i] + r1[i];
    if (x & 1) return i < dw - 1 ? (3 * s + 3 * r0[i + 1] + r1[i + 1] + 7) >> 4 : (4 * s + 7) >> 4;
    return i > 0 ? (3 * s + 3 * r0[i - 1] + r1[i - 1] + 8) >> 4 : (4 * s + 8) >> 4;
}

// the same eight upsampled chroma samples for an INTERIOR group (every neighbour exists): word loads, no edge tests
template <int HS, int VS>
__device__ __forceinline__ void chroma8_interior(const uint8_t *__restrict__ p, size_t stride, int rlo, int rhi, int x0, int y, int (&c)[8]) {
    auto six = [](const uint8_t *row, int i0, int (&s)[6]) {   // samples i0 - 1 .. i0 + 4 (i0 % 4 == 0)
        const uint32_t w = *reinterpret_cast<const uint32_t *>(row + i0);
        s[0] = row[i0 - 1];
        s[1] = w & 0xFF; s[2] = (w >> 8) & 0xFF; s[3] = (w >> 16) & 0xFF; s[4] = w >> 24;
        s[5] = row[i0 + 4];
    };
    if (HS == 1 && VS == 1) {
        const uint2 w = *reinterpret_cast<const uint2 *>(p + (size_t)y * stride + x0);
#pragma unroll
        for (int i = 0; i < 4; i++) { c[i] = (w.x >> (8 * i)) & 0xFF; c[4 + i] = (w.y >> (8 * i)) & 0xFF; }
    } else if (HS == 4) {
        const uint8_t *row = p + (size_t)y * stride + (x0 >> 2);
        const int s0 = row[0], s1 = row[1];
#pragma unroll
        for (int i = 0; i < 4; i++) { c[i] = s0; c[4 + i] = s1; }
    } else if (HS == 2 && VS == 1) {
        int s[6];
        six(p + (size_t)y * stride, x0 >> 1, s);
#pragma unroll
        for (int j = 0; j < 4; j++) {
            c[2 * j] = (3 * s[j + 1] + s[j] + 1) >> 2;
            c[2 * j + 1] = (3 * s[j + 1] + s[j + 2] + 2) >> 2;
        }
    } else if (HS == 1 && VS == 2) {
        const int r = y >> 1;
        const int rn = (y & 1) ? min(r + 1, rhi) : max(r - 1, rlo);
        const uint2 a = *reinterpret_cast<const uint2 *>(p + (size_t)r * stride + x0);
        const uint2 bq = *reinterpret_cast<const uint2 *>(p + (size_t)rn * stride + x0);
        const int bias = (y & 1) ? 2 : 1;
#pragma unroll
        for (int i = 0; i < 4; i++) {
            c[i] = (3 * (int)((a.x >> (8 * i)) & 0xFF) + (int)((bq.x >> (8 * i)) & 0xFF) + bias) >> 2;
            c[4 + i] = (3 * (int)((a.y >> (8 * i)) & 0xFF) + (int)((bq.y >> (8 * i)) & 0xFF) + bias) >> 2;
        }
    } else {   // h2v2
        const int r = y >> 1;
        const int rn = (y & 1) ? min(r + 1, rhi) : max(r - 1, rlo);
        int s0[6], s1[6], t[6];
        six(p + (size_t)r * stride, x0 >> 1, s0);
        six(p + (size_t)rn * stride, x0 >> 1, s1);
#pragma unroll
        for (int j = 0; j < 6; j++) t[j] = 3 * s0[j] + s1[j];
#pragma unroll
        for (int j = 0; j < 4; j++) {
            c[2 * j] = (3 * t[j + 1] + t[j] + 8) >> 4;
            c[2 * j + 1] = (3 * t[j + 1] + t[j + 2] + 7) >> 4;
        }
    }
}

template <int HS, int VS>
__global__ void __launch_bounds__(256)
k_upcolor(const uint8_t *__restrict__ py, const uint8_t *__restrict__ pcb, const uint8_t *__restrict__ pcr, Geom g,
          uint8_t *__restrict__ bgr, size_t step, int rlo, int rhi) {   // rlo / rhi: first / last chroma row the vertical filter may read
    const int gx = blockIdx.x * blockDim.x + threadIdx.x;  // group of 8 pixels
    const int y = blockIdx.y;
    const int x0 = gx * 8;
    if (x0 >= g.W) return;
    const size_t ys = (size_t)g.mcux * 8 * HS, cs = (size_t)g.mcux * 8;
    const int dw = g.dw[1];
    uint8_t *dst = bgr + (size_t)y * step + (size_t)x0 * 3;
    uint8_t o[24];
    // interior groups (all neighbours of all eight pixels exist, 8-byte aligned destination): vector loads and stores
    if (x0 >= 8 && x0 + 16 <= g.W && (reinterpret_cast<uintptr_t>(dst) & 7) == 0) {
        const uint2 yw = *reinterpret_cast<const uint2 *>(py + (size_t)y * ys + x0);
        int cbv[8], crv[8];
        uint32_t o32[6];
        chroma8_interior<HS, VS>(pcb, cs, rlo, rhi, x0, y, cbv);
        chroma8_interior<HS, VS>(pcr, cs, rlo, rhi, x0, y, crv);
        // jdcolor.c ycc_rgb_convert with the tables written out: r = y + ((91881 (cr - 128) + 32768) >> 16) etc. Here y sits
        // at bit 16 of the accumulator, the -128 and the rounding are one constant per channel, the sum is clamped to
        // [0, 255.99..] and the result is byte 2 of the word: same integers, a third fewer instructions per pixel.
        uint32_t B[8], G[8], R[8];
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const int Y16 = (int)__byte_perm(i < 4 ? yw.x : yw.y, 0u, 0x4044u | ((uint32_t)(i & 3) << 8));   // y << 16
            const int cb = cbv[i], cr = crv[i];
            const int r = 91881 * cr + Y16 + (32768 - 128 * 91881);
            const int b = 116130 * cb + Y16 + (32768 - 128 * 116130);
            const int gg = -22554 * cb - 46802 * cr + Y16 + (32768 + 128 * (22554 + 46802));
            R[i] = (uint32_t)min(0x00FFFFFF, max(0, r));
            B[i] = (uint32_t)min(0x00FFFFFF, max(0, b));
            G[i] = (uint32_t)min(0x00FFFFFF, max(0, gg));
        }
        // bytes b g r b | g r b g | r b g r per four pixels, every one byte 2 of its word
        uint2 *d2 = reinterpret_cast<uint2 *>(dst);
#pragma unroll
        for (int h = 0; h < 2; h++) {
            const int k = 4 * h;
            const uint32_t w0 = __byte_perm(__byte_perm(B[k], G[k], 0x0062), __byte_perm(R[k], B[k + 1], 0x0062), 0x5410);
            const uint32_t w1 = __byte_perm(__byte_perm(G[k + 1], R[k + 1], 0x0062), __byte_perm(B[k + 2], G[k + 2], 0x0062), 0x5410);
            const uint32_t w2 = __byte_perm(__byte_perm(R[k + 2], B[k + 3], 0x0062), __byte_perm(G[k + 3], R[k + 3], 0x0062), 0x5410);
            o32[3 * h] = w0; o32[3 * h + 1] = w1; o32[3 * h + 2] = w2;
        }
        d2[0] = make_uint2(o32[0], o32[1]);
        d2[1] = make_uint2(o32[2], o32[3]);
        d2[2] = make_uint2(o32[4], o32[5]);
        return;
    }
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const int x = min(x0 + i, g.W - 1);
        const int Y = py[(size_t)y * ys + x];
        const int cb = chroma_at<HS, VS>(pcb, cs, dw, rlo, rhi, x, y) - 128;
        const int cr = chroma_at<HS, VS>(pcr, cs, dw, rlo, rhi, x, y) - 128;
        const int r = Y + ((91881 * cr + 32768) >> 16);
        const int b = Y + ((116130 * cb + 32768) >> 16);
        const int gg = Y + ((-22554 * cb - 46802 * cr + 32768) >> 16);
        o[3 * i] = (uint8_t)min(255, max(0, b));
        o[3 * i + 1] = (uint8_t)min(255, max(0, gg));
        o[3 * i + 2] = (uint8_t)min(255, max(0, r));
    }
    const int nv = min(8, g.W - x0);
    for (int j = 0; j < nv * 3; j++) dst[j] = o[j];
}

// ------------------------------------------------------------------------------------------------------
size_t dec_sync_smem() { return sizeof(DecShared); }

cudaError_t launch_destuff(const uint8_t *in, size_t n, uint8_t *out, uint64_t *desc, uint32_t *ticket, int c0, int c1,
                           uint64_t *out_len, uint64_t *avail, uint32_t *bnd, uint32_t bnd_cap, uint32_t *nmark, uint32_t *err,
                           cudaStream_t s) {
    const int grid = std::max(1, std::min(148 * 4, c1 - c0));
    if (bnd) k_destuff<true><<<grid, 256, 0, s>>>(in, n, out, desc, ticket, c0, c1, out_len, avail, bnd, bnd_cap, nmark, err);
    else k_destuff<false><<<grid, 256, 0, s>>>(in, n, out, desc, ticket, c0, c1, out_len, avail, nullptr, 0, nullptr, err);
    return cudaGetLastError();
}

static cudaError_t dec_attr() {
    static std::atomic<uint64_t> done{0};   // one bit per device ordinal: the attribute is per device
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    const uint64_t bit = 1ull << (dev & 63);
    if (done.load(std::memory_order_acquire) & bit) return cudaSuccess;
    e = cudaFuncSetAttribute(k_dec_sync<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(DecShared));
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(k_dec_sync<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(DecShared));
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(k_dec_write<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(DecWriteShared));
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(k_dec_write<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(DecWriteShared));
    if (e != cudaSuccess) return e;
    done.fetch_or(bit, std::memory_order_release);
    return cudaSuccess;
}

cudaError_t launch_dec_sync(const uint8_t *u, const uint64_t *u_len, const void *tb, uint64_t *st_in, uint64_t *st_out,
                            uint32_t *nblk, int bpm, int hv, int inner, int mode, uint8_t *done, uint32_t *changed,
                            size_t nsub, const uint32_t *bnd, const uint32_t *nmark, const uint32_t *skip_if_zero, cudaStream_t s) {
    cudaError_t e = dec_attr();
    if (e != cudaSuccess) return e;
    const unsigned grid = (unsigned)((nsub + DEC_THREADS - 1) / DEC_THREADS);
    if (grid == 0) return cudaSuccess;
    if (bnd) k_dec_sync<true><<<grid, DEC_THREADS, sizeof(DecShared), s>>>(u, u_len, (const DecTables *)tb, st_in, st_out, nblk, bpm, hv,
                                                                        inner, mode, done, changed, bnd, nmark, skip_if_zero);
    else k_dec_sync<false><<<grid, DEC_THREADS, sizeof(DecShared), s>>>(u, u_len, (const DecTables *)tb, st_in, st_out, nblk, bpm, hv,
                                                                     inner, mode, done, changed, nullptr, nullptr, skip_if_zero);
    return cudaGetLastError();
}

cudaError_t launch_dec_sync_long(const uint8_t *u, const uint64_t *u_len, const void *tb, uint64_t *st_in, uint64_t *st_out,
                                 uint32_t *nblk, int bpm, int hv, int first, int group, uint32_t *changed, size_t nsub,
                                 const uint32_t *bnd, const uint32_t *nmark, cudaStream_t s) {
    const int DEC_GROUP = group < 1 ? 1 : group;
    const size_t ngrp = (nsub + DEC_GROUP - 1) / DEC_GROUP;
    const unsigned grid = (unsigned)((ngrp + DEC_LONG_THREADS - 1) / DEC_LONG_THREADS);
    if (grid == 0) return cudaSuccess;
    if (bnd) k_dec_sync_long<true><<<grid, DEC_LONG_THREADS, 0, s>>>(u, u_len, (const DecTables *)tb, st_in, st_out, nblk, bpm, hv, first, DEC_GROUP, changed, bnd, nmark);
    else k_dec_sync_long<false><<<grid, DEC_LONG_THREADS, 0, s>>>(u, u_len, (const DecTables *)tb, st_in, st_out, nblk, bpm, hv, first, DEC_GROUP, changed, nullptr, nullptr);
    return cudaGetLastError();
}

cudaError_t launch_dec_write(const uint8_t *u, const uint64_t *u_len, const void *tb, const uint64_t *st_out,
                             const uint32_t *blk_start, int bpm, int hv, int16_t *coef, int16_t *dcarr, uint32_t nblocks,
                             uint32_t *err, size_t nsub_max, const uint32_t *bnd, const uint32_t *nmark, cudaStream_t s) {
    cudaError_t e = dec_attr();
    if (e != cudaSuccess) return e;
    const unsigned grid = (unsigned)((nsub_max + DEC_THREADS - 1) / DEC_THREADS);
    if (bnd) k_dec_write<true><<<grid, DEC_THREADS, sizeof(DecWriteShared), s>>>(u, u_len, (const DecTables *)tb, st_out, blk_start, bpm,
                                                                              hv, coef, dcarr, nblocks, err, bnd, nmark);
    else k_dec_write<false><<<grid, DEC_THREADS, sizeof(DecWriteShared), s>>>(u, u_len, (const DecTables *)tb, st_out, blk_start, bpm,
                                                                           hv, coef, dcarr, nblocks, err, nullptr, nullptr);
    return cudaGetLastError();
}

cudaError_t launch_scan_u32(const uint32_t *in, uint32_t *out, size_t n, uint64_t *desc, uint32_t *ticket, uint32_t *err,
                            cudaStream_t s) {
    k_scan_u32<<<148 * 4, 256, 0, s>>>(in, out, n, desc, ticket, err);
    return cudaGetLastError();
}

cudaError_t launch_dc_scan(int16_t *coef, const Geom &g, int ncomp, uint64_t *desc, uint32_t *ticket, size_t desc_stride,
                           uint32_t *err, cudaStream_t s) {
    dim3 grid(148 * 2, ncomp);
    k_dc_scan<<<grid, 256, 0, s>>>(coef, g.bpm, g.hs * g.vs, (size_t)g.mcux * g.mcuy, desc, ticket, desc_stride, err);
    return cudaGetLastError();
}

template <bool GRAY>
static cudaError_t idct_launch(const int16_t *coef, const int16_t *dcarr, const Geom &g, const void *tb, uint8_t *py, uint8_t *pcb,
                               uint8_t *pcr, int rst_mcus, size_t out_step, cudaStream_t s) {
    // the dynamic shared-memory attribute is per device: one bit per device ordinal
    static std::atomic<uint64_t> attr_done{0};
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    const uint64_t bit = 1ull << (dev & 63);
    if (!(attr_done.load(std::memory_order_acquire) & bit)) {
        e = cudaFuncSetAttribute(k_idct<GRAY>, cudaFuncAttributeMaxDynamicSharedMemorySize, IDCT_SMEM);
        if (e != cudaSuccess) return e;
        attr_done.fetch_or(bit, std::memory_order_release);
    }
    const int ntile = (g.nblocks + IDCT_TILE - 1) / IDCT_TILE;
    k_idct<GRAY><<<std::max(1, std::min(ntile, 148 * 2)), 256, IDCT_SMEM, s>>>(coef, dcarr, g, (const DecTables *)tb, py, pcb, pcr,
                                                                               rst_mcus, out_step);
    return cudaGetLastError();
}

cudaError_t launch_idct(const int16_t *coef, const int16_t *dcarr, const Geom &g, const void *tb, uint8_t *py, uint8_t *pcb,
                        uint8_t *pcr, int rst_mcus, cudaStream_t s) {
    return idct_launch<false>(coef, dcarr, g, tb, py, pcb, pcr, rst_mcus, 0, s);
}

cudaError_t launch_idct_gray(const int16_t *coef, const int16_t *dcarr, const Geom &g, const void *tb, uint8_t *gray, size_t step,
                             int rst_mcus, cudaStream_t s) {
    return idct_launch<true>(coef, dcarr, g, tb, gray, nullptr, nullptr, rst_mcus, step, s);
}

template <int HS, int VS>
static cudaError_t upcolor_one(const uint8_t *py, const uint8_t *pcb, const uint8_t *pcr, const Geom &g, uint8_t *bgr,
                               size_t step, int halo_top, int halo_bottom, cudaStream_t s) {
    dim3 grid(((g.W + 7) / 8 + 255) / 256, g.H);
    k_upcolor<HS, VS><<<grid, 256, 0, s>>>(py, pcb, pcr, g, bgr, step, halo_top ? -1 : 0, halo_bottom ? g.dh[1] : g.dh[1] - 1);
    return cudaGetLastError();
}

cudaError_t launch_upcolor(const uint8_t *py, const uint8_t *pcb, const uint8_t *pcr, const Geom &g, uint8_t *bgr, size_t step,
                           cudaStream_t s, int halo_top, int halo_bottom) {
    if (g.hs == 1 && g.vs == 1) return upcolor_one<1, 1>(py, pcb, pcr, g, bgr, step, halo_top, halo_bottom, s);
    if (g.hs == 2 && g.vs == 1) return upcolor_one<2, 1>(py, pcb, pcr, g, bgr, step, halo_top, halo_bottom, s);
    if (g.hs == 1 && g.vs == 2) return upcolor_one<1, 2>(py, pcb, pcr, g, bgr, step, halo_top, halo_bottom, s);
    if (g.hs == 2 && g.vs == 2) return upcolor_one<2, 2>(py, pcb, pcr, g, bgr, step, halo_top, halo_bottom, s);
    if (g.hs == 4 && g.vs == 1) return upcolor_one<4, 1>(py, pcb, pcr, g, bgr, step, halo_top, halo_bottom, s);
    return cudaErrorInvalidValue;
}

}  // namespace b2j
