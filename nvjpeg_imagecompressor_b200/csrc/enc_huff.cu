// enc_huff.cu -- optimized-Huffman table generation, entropy coding (pack), tile scan and byte stuffing.
//
// Replaces the second half of nvjpegEncodeImage (reference call site ImageCompressorImpl.cu:280; nvJPEG kernels
// GenerateOptimizeHuffmanTableKernel / BlockLengthKernel / SumBlocksKernel / BlockAssembleKernel /
// ByteStuffingKernel, SURVEY.md 2b) and nvjpegEncodeRetrieveBitstream's header writing (:285-287).
// Algorithms follow libjpeg-turbo jchuff.c (jpeg_gen_optimal_table, encode_one_block) and jcmarker.c as
// restated in SURVEY.md Appendix A.6-A.8, bit-exactly (checked by tests/ against the CPU checker).
#include "common.cuh"
#include "kernels.h"

namespace b2j {

// ------------------------------------------------------------------------------------------------------
// Annex K.3-K.6 standard tables (jcparam.c std_huff_tables)
__constant__ uint8_t c_std_bits[4][17] = {
    {0, 0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0},
    {0, 0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 0x7d},
    {0, 0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0},
    {0, 0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 0x77}};
__constant__ uint8_t c_std_dc_val[12] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11};
__constant__ uint8_t c_std_ac_val[2][162] = {
    {0x01, 0x02, 0x03, 0x00, 0x04, 0x11, 0x05, 0x12, 0x21, 0x31, 0x41, 0x06, 0x13, 0x51, 0x61, 0x07, 0x22, 0x71,
     0x14, 0x32, 0x81, 0x91, 0xa1, 0x08, 0x23, 0x42, 0xb1, 0xc1, 0x15, 0x52, 0xd1, 0xf0, 0x24, 0x33, 0x62, 0x72,
     0x82, 0x09, 0x0a, 0x16, 0x17, 0x18, 0x19, 0x1a, 0x25, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x34, 0x35, 0x36, 0x37,
     0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59,
     0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a, 0x83,
     0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a, 0xa2, 0xa3,
     0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3,
     0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe1, 0xe2,
     0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf1, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa},
    {0x00, 0x01, 0x02, 0x03, 0x11, 0x04, 0x05, 0x21, 0x31, 0x06, 0x12, 0x41, 0x51, 0x07, 0x61, 0x71, 0x13, 0x22,
     0x32, 0x81, 0x08, 0x14, 0x42, 0x91, 0xa1, 0xb1, 0xc1, 0x09, 0x23, 0x33, 0x52, 0xf0, 0x15, 0x62, 0x72, 0xd1,
     0x0a, 0x16, 0x24, 0x34, 0xe1, 0x25, 0xf1, 0x17, 0x18, 0x19, 0x1a, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x35, 0x36,
     0x37, 0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58,
     0x59, 0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a,
     0x82, 0x83, 0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a,
     0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba,
     0xc2, 0xc3, 0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda,
     0xe2, 0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa}};

// ------------------------------------------------------------------------------------------------------
// k_tables: one CTA, warp t builds table t (DC0, AC0, DC1, AC1), then the JFIF headers are written. NC = 1 (gray):
// only DC0 / AC0 are coded; warps 2 and 3 load the standard chroma tables (never emitted, never looked up) instead of
// building codes from the all-zero DC1 / AC1 histograms, and the headers have one DQT, two DHTs and one component.
//
// jpeg_gen_optimal_table, warp-parallel: lane l owns symbols l, l+32, ... (9 per lane, symbol 256 = the reserved
// all-ones code point). Each merge step finds c1 = least non-zero frequency with ties to the LARGER index, c2 = next
// least, by two warp reductions each (min of frequency, then max of index among the minima); tree membership is a
// group id per symbol so "increment codesize along the others chain" becomes "increment every member".
template <int NC>
__global__ void __launch_bounds__(128)
k_tables(const uint32_t *hist /* the predecessor's output: no __restrict__, loads must stay behind pdl_wait() */, int optimize,
         HuffDev *__restrict__ huff, const QuantDev *__restrict__ qd,
         int full_w, int full_h, int hs, int vs, uint8_t *__restrict__ out, int emit_header, int restart_interval,
         uint32_t *__restrict__ err_out) {
    __shared__ uint8_t s_bits[4][17];
    __shared__ uint8_t s_vals[4][256];
    __shared__ uint32_t s_enc[4][256];
    __shared__ int s_cs[4][257];
    __shared__ int s_cnt[4][33];
    __shared__ int s_base[4][33];
    __shared__ uint32_t s_nsym[4];
    __shared__ uint32_t s_err;
    __shared__ uint8_t s_hdr[1024];
    __shared__ uint32_t s_hdr_len;
    const int t = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const unsigned FULL = 0xffffffffu;
    pdl_trigger();   // k_pack's CTAs clear their buffers meanwhile
    if (threadIdx.x == 0) s_err = 0;
    for (int i = lane; i < 256; i += 32) { s_vals[t][i] = 0; s_enc[t][i] = 0; }
    __syncthreads();
    pdl_wait();

    if (!optimize || (NC == 1 && t >= 2)) {
        if (lane < 17) s_bits[t][lane] = c_std_bits[t][lane];
        const int ns = (t & 1) ? 162 : 12;
        for (int i = lane; i < ns; i += 32) s_vals[t][i] = (t & 1) ? c_std_ac_val[t >> 1][i] : c_std_dc_val[i];
        if (lane == 0) s_nsym[t] = ns;
    } else {
        uint32_t f[9];
        int cs[9], grp[9];
#pragma unroll
        for (int j = 0; j < 9; j++) {
            const int i = lane + 32 * j;
            f[j] = i < 256 ? hist[t * 257 + i] : (i == 256 ? 1u : 0u);
            cs[j] = 0;
            grp[j] = i;
        }
        // Fast selection while the two least frequencies are below 2^23: one 32-bit key per symbol, frequency in the
        // upper 23 bits and (511 - index) below it, so "least frequency, ties to the larger index" is one REDUX.MIN;
        // the lane that owned c1 offers its second-best key for c2. Larger frequencies take the four-reduction path.
        constexpr uint32_t KEY_NONE = 0xffffffffu;
        uint32_t key[9];
#pragma unroll
        for (int j = 0; j < 9; j++) {
            const int i = lane + 32 * j;
            key[j] = (f[j] != 0 && f[j] < (1u << 23)) ? ((f[j] << 9) | (uint32_t)(511 - i)) : KEY_NONE;
        }
        for (int iter = 0; iter < 300; iter++) {
            // this lane's two smallest keys: a tournament (depth 7) instead of a 9-step insertion chain (depth 18),
            // the loop is one long dependency chain per table
            uint32_t b1, b2;
            {
                const uint32_t l01 = min(key[0], key[1]), h01 = max(key[0], key[1]);
                const uint32_t l23 = min(key[2], key[3]), h23 = max(key[2], key[3]);
                const uint32_t l45 = min(key[4], key[5]), h45 = max(key[4], key[5]);
                const uint32_t l67 = min(key[6], key[7]), h67 = max(key[6], key[7]);
                const uint32_t a1 = min(l01, l23), a2 = min(max(l01, l23), min(h01, h23));
                const uint32_t c1 = min(l45, l67), c2 = min(max(l45, l67), min(h45, h67));
                const uint32_t d1 = min(a1, c1), d2 = min(max(a1, c1), min(a2, c2));
                b1 = min(d1, key[8]);
                b2 = min(max(d1, key[8]), d2);
            }
            const uint32_t k1 = __reduce_min_sync(FULL, b1);
            const uint32_t k2 = k1 == KEY_NONE ? KEY_NONE : __reduce_min_sync(FULL, b1 == k1 ? b2 : b1);
            uint32_t m1, m2;
            int c1, c2;
            if (k2 != KEY_NONE) {
                m1 = k1 >> 9; c1 = 511 - (int)(k1 & 511u);
                m2 = k2 >> 9; c2 = 511 - (int)(k2 & 511u);
            } else {
                // c1
                uint32_t bf = 0xffffffffu;
                int bi = -1;
#pragma unroll
                for (int j = 0; j < 9; j++)
                    if (f[j] != 0 && f[j] <= 1000000000u && f[j] <= bf) { bf = f[j]; bi = lane + 32 * j; }
                m1 = __reduce_min_sync(FULL, bf);
                if (m1 == 0xffffffffu) break;
                c1 = __reduce_max_sync(FULL, bf == m1 ? bi : -1);
                // c2
                bf = 0xffffffffu;
                bi = -1;
#pragma unroll
                for (int j = 0; j < 9; j++)
                    if (f[j] != 0 && f[j] <= 1000000000u && f[j] <= bf && (lane + 32 * j) != c1) { bf = f[j]; bi = lane + 32 * j; }
                m2 = __reduce_min_sync(FULL, bf);
                if (m2 == 0xffffffffu) break;
                c2 = __reduce_max_sync(FULL, bf == m2 ? bi : -1);
            }
#pragma unroll
            for (int j = 0; j < 9; j++) {
                const int i = lane + 32 * j;
                if (i == c1) {
                    f[j] = m1 + m2;
                    key[j] = f[j] < (1u << 23) ? ((f[j] << 9) | (uint32_t)(511 - i)) : KEY_NONE;
                }
                if (i == c2) { f[j] = 0; key[j] = KEY_NONE; }
                if (i <= 256 && (grp[j] == c1 || grp[j] == c2) && (cs[j] > 0 || i == c1 || i == c2)) {
                    cs[j]++;
                    grp[j] = c1;
                }
            }
        }
        for (int l = lane; l < 33; l += 32) s_cnt[t][l] = 0;
        __syncwarp();
#pragma unroll
        for (int j = 0; j < 9; j++) {
            const int i = lane + 32 * j;
            if (i <= 256) {
                s_cs[t][i] = cs[j];
                if (cs[j] > 32) s_err = 2;
                else if (cs[j] > 0) atomicAdd(&s_cnt[t][cs[j]], 1);
            }
        }
        __syncwarp();
        // huffval: symbols 0..255 sorted by (natural codesize, symbol). First slot of every codesize from the counts
        // (taken before the length limiting below rewrites them; the reserved symbol 256 holds no slot), then per 32
        // symbols the lanes of equal codesize rank themselves with MATCH.ANY.
        {
            const int l = lane + 1;   // codesize 1..32
            const int n = s_cnt[t][l] - (s_cs[t][256] == l ? 1 : 0);
            int inc = n;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int y = __shfl_up_sync(FULL, inc, o);
                if (lane >= o) inc += y;
            }
            s_base[t][l] = inc - n;
            if (lane == 31) s_nsym[t] = (uint32_t)inc;
        }
        __syncwarp();
        if (lane == 0) {
            int *bits = s_cnt[t];
            for (int i = 32; i > 16; i--)
                while (bits[i] > 0) {
                    int j = i - 2;
                    while (bits[j] == 0) j--;
                    bits[i] -= 2;
                    bits[i - 1]++;
                    bits[j + 1] += 2;
                    bits[j]--;
                }
            int i = 16;
            while (bits[i] == 0) i--;
            bits[i]--;
            s_bits[t][0] = 0;
            for (int l = 1; l <= 16; l++) s_bits[t][l] = (uint8_t)bits[l];
        }
        // huffval, second half: per 32 symbols the lanes of equal codesize rank themselves with MATCH.ANY
        for (int c = 0; c < 8; c++) {
            const int sym = c * 32 + lane;
            const int v = s_cs[t][sym] <= 32 ? s_cs[t][sym] : 0;   // > 32: error already flagged (s_err = 2)
            const unsigned same = __match_any_sync(FULL, v);
            const int base = v > 0 ? s_base[t][v] : 0;
            __syncwarp();
            if (v > 0) {
                s_vals[t][base + __popc(same & ((1u << lane) - 1u))] = (uint8_t)sym;
                if ((same & ((1u << lane) - 1u)) == 0) s_base[t][v] = base + __popc(same);
            }
            __syncwarp();
        }
    }
    __syncwarp();
    // Annex C code assignment: lane l (1..16) derives the first code and the first huffval index of length l from
    // the counts, then every lane assigns the codes of its huffval positions
    {
        int cnt = (lane >= 1 && lane <= 16) ? (int)s_bits[t][lane] : 0;
        int first_idx = cnt;   // exclusive prefix of the counts
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_up_sync(FULL, first_idx, o);
            if (lane >= o) first_idx += y;
        }
        first_idx -= cnt;
        // first code of length l: code(l) = (code(l-1) + count(l-1)) << 1, code(1) = 0
        uint32_t fc = 0;
        for (int l = 2; l <= 16; l++) {
            const uint32_t prev_cnt = (uint32_t)__shfl_sync(FULL, cnt, l - 1);
            const uint32_t prev_fc = __shfl_sync(FULL, fc, l - 1);
            if (lane == l) fc = (prev_fc + prev_cnt) << 1;
        }
        s_cs[t][lane] = first_idx;         // reuse: [0..31] first index, [32..63] first code (s_cs is dead here)
        s_cs[t][32 + lane] = (int)fc;
        __syncwarp();
        const int ns = (int)s_nsym[t];
        for (int p = lane; p < ns; p += 32) {
            // length of position p: the largest l with first_idx(l) <= p among the lengths that have codes
            int l = 1;
#pragma unroll 1
            for (int q = 1; q <= 16; q++)
                if (s_bits[t][q] != 0 && s_cs[t][q] <= p) l = q;
            const uint32_t code = (uint32_t)s_cs[t][32 + l] + (uint32_t)(p - s_cs[t][l]);
            s_enc[t][s_vals[t][p]] = (code << 8) | (uint32_t)l;
        }
    }
    __syncthreads();

    // ---- headers (jcmarker.c): SOI, JFIF APP0, 2 x DQT, SOF0, 4 x DHT, SOS (gray: 1 x DQT, 2 x DHT) -- section offsets by thread 0, bytes by
    //      all threads
    __shared__ uint32_t s_off[9];   // DQT0, DQT1, SOF0, DHT0..3, SOS, DRI (jcmarker.c: after the scan's DHTs, before SOS)
    constexpr int NH = NC == 1 ? 2 : 4;   // DHTs
    if (threadIdx.x == 0) {
        uint32_t n = 20;
        s_off[0] = n; n += 69;
        if (NC == 3) { s_off[1] = n; n += 69; }
        s_off[2] = n; n += 10 + 3 * NC;
        for (int q = 0; q < NH; q++) { s_off[3 + q] = n; n += 21 + s_nsym[q]; }
        s_off[8] = n; if (restart_interval) n += 6;
        s_off[7] = n; n += 8 + 2 * NC;
        if (!emit_header) n = 0;
        s_hdr_len = n;
        huff->hdr_len = n;
        huff->err = s_err;
        *err_out = s_err;
    }
    __syncthreads();
    if (emit_header) {
        uint8_t *h = s_hdr;
        const int x = threadIdx.x;
        if (x < 20) {
            const uint8_t app0[20] = {0xFF, 0xD8, 0xFF, 0xE0, 0, 16, 'J', 'F', 'I', 'F', 0, 1, 1, 0, 0, 1, 0, 1, 0, 0};
            h[x] = app0[x];
        }
        if (NC == 3 || x < 64) {   // DQT: thread x -> table x >> 6, coefficient x & 63 (zig-zag order)
            const int q = x >> 6, k = x & 63;
            uint8_t *d = h + s_off[q];
            if (k == 0) { d[0] = 0xFF; d[1] = 0xDB; d[2] = 0; d[3] = 67; d[4] = (uint8_t)q; }
            d[5 + k] = (uint8_t)qd->q[q][zigzag_nat_rt(k)];
        }
        if (x == 32) {
            uint8_t *d = h + s_off[2];
            if constexpr (NC == 1) {
                const uint8_t sof[13] = {0xFF, 0xC0, 0, 11, 8, (uint8_t)(full_h >> 8), (uint8_t)full_h, (uint8_t)(full_w >> 8), (uint8_t)full_w,
                                         1, 1, 0x11, 0};
                for (int i = 0; i < 13; i++) d[i] = sof[i];
            } else {
                const uint8_t sof[19] = {0xFF, 0xC0, 0, 17, 8, (uint8_t)(full_h >> 8), (uint8_t)full_h, (uint8_t)(full_w >> 8), (uint8_t)full_w,
                                         3, 1, (uint8_t)((hs << 4) | vs), 0, 2, 0x11, 1, 3, 0x11, 1};
                for (int i = 0; i < 19; i++) d[i] = sof[i];
            }
        }
        if (x == 96 && restart_interval) {
            uint8_t *d = h + s_off[8];
            d[0] = 0xFF; d[1] = 0xDD; d[2] = 0; d[3] = 4; d[4] = (uint8_t)(restart_interval >> 8); d[5] = (uint8_t)restart_interval;
        }
        if (x == 64) {
            uint8_t *d = h + s_off[7];
            if constexpr (NC == 1) {
                const uint8_t sos[10] = {0xFF, 0xDA, 0, 8, 1, 1, 0x00, 0, 63, 0};
                for (int i = 0; i < 10; i++) d[i] = sos[i];
            } else {
                const uint8_t sos[14] = {0xFF, 0xDA, 0, 12, 3, 1, 0x00, 2, 0x11, 3, 0x11, 0, 63, 0};
                for (int i = 0; i < 14; i++) d[i] = sos[i];
            }
        }
        if (NC == 3 || x < 64) {   // DHT q by warp q
            const int q = x >> 5;
            const int ns = (int)s_nsym[q];
            uint8_t *d = h + s_off[3 + q];
            const uint8_t tcth[4] = {0x00, 0x10, 0x01, 0x11};
            if (lane == 0) { d[0] = 0xFF; d[1] = 0xC4; d[2] = (uint8_t)((19 + ns) >> 8); d[3] = (uint8_t)(19 + ns); d[4] = tcth[q]; }
            if (lane >= 1 && lane <= 16) d[4 + lane] = s_bits[q][lane];
            for (int i = lane; i < ns; i += 32) d[21 + i] = s_vals[q][i];
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < (int)s_hdr_len; i += 128) out[i] = s_hdr[i];
    for (int i = threadIdx.x; i < 1024; i += 128) {
        huff->enc[i >> 8][i & 255] = s_enc[i >> 8][i & 255];
        huff->vals[i >> 8][i & 255] = s_vals[i >> 8][i & 255];
    }
    if (threadIdx.x < 68) huff->bits[threadIdx.x / 17][threadIdx.x % 17] = s_bits[threadIdx.x / 17][threadIdx.x % 17];
    if (threadIdx.x < 4) huff->nsym[threadIdx.x] = s_nsym[threadIdx.x];
}

// ------------------------------------------------------------------------------------------------------
// k_pack: token-parallel entropy coding (jchuff.c encode_one_block's emit_bits, without its run-length walk: that
// happened once, in k_fdct). Persistent CTAs of PACK_WARPS warps walk the fdct tiles; all the work is convergent and
// every token is looked up ONCE:
//   1. warp w takes a contiguous share of the tile's token run; every lane loads PACK_K consecutive tokens per step
//      (16-byte loads); a warp scan of the lanes' bit counts gives every lane its bit position inside the share; the
//      lane appends its codes to a 64-bit accumulator and ORs every completed 32-bit word into the warp's own bit
//      buffer, which starts at bit 0 (predicated red.shared: the words at a lane's ends are shared with its
//      neighbours). The share's length falls out of the walk.
//   2. one CTA barrier: the warps' lengths give each share its bit offset inside the tile and the tile's size
//   3. every warp shifts its buffer into place on the way out: words wholly inside its bit range go straight to the
//      tile's fixed-size slot in global memory (tile t at t*SLOT_WORDS); the word it shares with a neighbour is
//      OR-ed into a per-boundary cell that thread 0 writes after the NEXT tile's barrier (cells double-buffered)
// Dense tiles (more tokens than the warp buffers are sure to hold, or a buffer that overflowed) take the two-pass
// path: lengths first, then the bits are scattered window by window into one tile-wide buffer.
// Raw-DC tokens were resolved by k_dc_edge_hist; ZRL prefixes (token bits 27:26) ride on the token when there is one and
// the bits fit a word, and are emitted in a side branch otherwise.
constexpr int WIN_WORDS = 2048;                  // dense tiles: 64 kbit window of the tile's bit string
constexpr int SUB_WORDS = 512;                   // per-warp bit buffer: 16 kbit (a typical share is ~7.5 kbit)
constexpr int PACK_THREADS = 128;                // one CTA per tile at a time, PACK_WARPS contiguous shares
constexpr int PACK_WARPS = PACK_THREADS / 32;
constexpr int PACK_CTAS = 8;                     // resident CTAs per SM (register budget)
constexpr int PACK_K = 8;                        // consecutive tokens per lane and step
constexpr int PACK_STEP = 32 * PACK_K;           // tokens per warp and step
constexpr uint32_t PACK_DENSE_TOKENS = 7000;     // above this the shares may not fit the warp buffers: two-pass path
constexpr uint32_t TOK_NULL = ((1u << 6) | 3u) << 16;   // bin (run 1, size 0, tcode 2 = DC luma): no such symbol -> no code, no bits
static_assert(bin_table(TOK_NULL >> 16) == 0u, "TOK_NULL must name a DC table with a run");

struct PackShared {
    uint32_t buf[WIN_WORDS];
    uint32_t sub[PACK_WARPS][SUB_WORDS + 4];
    uint32_t code[1024];                         // [token bits 25:16] code << size (the value bits are OR-ed below it)
    uint8_t len[4096];                           // [token bits 27:16] code length + size + ZRL count * length of the ZRL code
    uint32_t wlen[3][PACK_WARPS];                // bit counts of the warps' shares, three tiles deep
    uint32_t bnd[2][PACK_WARPS + 1];             // words shared by two shares (cell b: the word holding the start of share b)
};

// One lane's contiguous piece of the bit string: bits are appended to a 64-bit accumulator and every completed
// 32-bit word goes to the buffer. `cnt` = valid low bits of acc that are not flushed yet (< 32 between calls).
// WINDOWED (dense tiles, the warps share one window): atomicOr, words outside the window [0, nwords) are skipped.
// Otherwise (the warp's own buffer): a word is completed by exactly one lane, which stores it whole -- bits that
// earlier lanes own in it are zero in that store and are OR-ed in afterwards (finish(), after a warp barrier), so
// the hot path has no atomics and the buffer needs no clearing except the word a share ends in. Words at or beyond
// the byte address `limit` are dropped (the caller notices the overflow from the share's length).
template <bool WINDOWED>
struct LaneEmitter {
    uint64_t acc;
    uint32_t cnt;
    uint32_t addr, limit;   // fast: shared byte address of the current word / end of the buffer
    int wi;                 // windowed: word index relative to the window
    uint32_t win;           // windowed: words in the window
    uint32_t *buf;
    __device__ __forceinline__ void start(uint32_t *b, int pos, uint32_t nwords) {
        buf = b; acc = 0; cnt = (uint32_t)pos & 31u; wi = pos >> 5; win = nwords;
        addr = smem_u32(b) + (uint32_t)(pos >> 5) * 4u;
        limit = smem_u32(b) + nwords * 4u;
    }
    __device__ __forceinline__ void put(uint32_t bits, uint32_t n) {   // n <= 32
        acc = (acc << n) | bits;
        cnt += n;
        if (WINDOWED) {
            if (cnt >= 32u) {
                cnt -= 32u;
                if ((uint32_t)wi < win) atomicOr(&buf[wi], (uint32_t)(acc >> cnt));
                wi++;
            }
        } else {
            const uint32_t wv = __funnelshift_r((uint32_t)acc, (uint32_t)(acc >> 32), cnt);   // acc >> (cnt - 32) if cnt >= 32
            asm volatile("{\n\t.reg .pred p, q;\n\tsetp.ge.u32 p, %1, 32;\n\tsetp.lt.and.u32 q, %0, %3, p;\n\t"
                         "@q st.shared.b32 [%0], %2;\n\t@p add.u32 %0, %0, 4;\n\t@p sub.u32 %1, %1, 32;\n\t}"
                         : "+r"(addr), "+r"(cnt) : "r"(wv), "r"(limit) : "memory");
        }
    }
    __device__ __forceinline__ void finish() {
        if (cnt) {
            const uint32_t wv = (uint32_t)acc << (32u - cnt);
            if (WINDOWED) { if ((uint32_t)wi < win) atomicOr(&buf[wi], wv); }
            else if (addr < limit) atomicOr(buf + ((addr - smem_u32(buf)) >> 2), wv);
        }
    }
};

// PACK_K tokens of one lane: virtual indices [v0, v0 + PACK_K) of the walk that starts at the 16-byte boundary
// below the tile's run; indices outside [a, hi) become TOK_NULL
__device__ __forceinline__ void load_tokens(const uint4 *tk4, uint32_t v0, uint32_t a, uint32_t hi, uint32_t (&w)[PACK_K]) {
#pragma unroll
    for (int q = 0; q < PACK_K / 4; q++) {
        const uint4 x = __ldg(tk4 + (v0 >> 2) + q);
        w[4 * q] = x.x; w[4 * q + 1] = x.y; w[4 * q + 2] = x.z; w[4 * q + 3] = x.w;
    }
    if (v0 < a || v0 + PACK_K > hi) {
#pragma unroll
        for (int k = 0; k < PACK_K; k++)
            if (v0 + k < a || v0 + k >= hi) w[k] = TOK_NULL;
    }
}

// The warp's share [lo, hi) of the walk, coded into `buf` starting at bit `run`; returns the bit position after it.
template <bool WINDOWED>
__device__ __forceinline__ int pack_scatter(const PackShared &sh, uint32_t *buf, uint32_t nwords, const uint4 *tk4, uint32_t a,
                                            uint32_t lo, uint32_t hi, int run, int lane, uint32_t zr_y, uint32_t zr_c) {
    for (uint32_t s0 = lo; s0 < hi; s0 += PACK_STEP) {
        const uint32_t v0 = s0 + lane * PACK_K;
        uint32_t w[PACK_K], L[PACK_K], bits[PACK_K];
        uint32_t Lt = 0;
        if (v0 < hi) load_tokens(tk4, v0, a, hi, w);
        else {
#pragma unroll
            for (int k = 0; k < PACK_K; k++) w[k] = TOK_NULL;
        }
#pragma unroll
        for (int k = 0; k < PACK_K; k++) {
            const uint32_t i12 = (w[k] >> 16) & 0xFFFu;
            L[k] = sh.len[i12];
            bits[k] = sh.code[i12 & 0x3FFu] | (w[k] & 0xFFFFu);
            Lt += L[k];
        }
        uint32_t inc = Lt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += y;
        }
        LaneEmitter<WINDOWED> e;
        e.start(buf, run + (int)(inc - Lt), nwords);
        if (!WINDOWED) {
            // lane 0 continues the word the previous step ended in: it takes the bits that are already there
            if (lane == 0 && e.cnt != 0u && e.addr < e.limit) e.acc = (uint64_t)(buf[run >> 5] >> (32u - e.cnt));
        }
        run += (int)__shfl_sync(0xffffffffu, inc, 31);
#pragma unroll
        for (int k = 0; k < PACK_K; k++) {
            uint32_t n = L[k];
            const uint32_t nz = (w[k] >> 26) & 3u;
            uint32_t b = bits[k];
            if (nz) {   // ZRL symbols ahead of this coefficient (about one token in sixty, i.e. one lane in most steps)
                // AC tokens: tcode 0 luma / 1 chroma, and the table field holds (tcode + run) & 3 (common.cuh)
                const uint32_t zr = (((w[k] >> 16) - (w[k] >> 22)) & 1u) ? zr_c : zr_y;
                const uint32_t zl = zr & 31u, tl = n - nz * zl;
                if (nz == 1u && n <= 32u) {   // the usual case: the ZRL code rides on top of the token's bits
                    b |= (zr >> 8) << tl;
                } else {
                    n = tl;
                    e.put(zr >> 8, zl);
                    if (nz > 1u) {
                        e.put(zr >> 8, zl);
                        if (nz > 2u) e.put(zr >> 8, zl);
                    }
                }
            }
            e.put(b, n);
        }
        if (!WINDOWED) __syncwarp();   // every whole word of this step is stored: now the pieces that do not fill a word
        e.finish();
        if (!WINDOWED) __syncwarp();
    }
    return run;
}

// bits of the warp's share without coding them (two-pass path)
__device__ __forceinline__ uint32_t pack_length(const PackShared &sh, const uint4 *tk4, uint32_t a, uint32_t lo, uint32_t hi, int lane) {
    uint32_t len = 0;
    for (uint32_t v0 = lo + lane * PACK_K; v0 < hi; v0 += PACK_STEP) {
        uint32_t w[PACK_K];
        load_tokens(tk4, v0, a, hi, w);
#pragma unroll
        for (int k = 0; k < PACK_K; k++) len += sh.len[(w[k] >> 16) & 0xFFFu];
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) len += __shfl_xor_sync(0xffffffffu, len, o);
    return len;
}

// the previous tile's shared words: cell b holds the bits of the word that contains the start of share b (and the end
// of share b - 1); consecutive cells can name the same word when a share is shorter than a word
__device__ __forceinline__ void pack_flush_shared_words(uint32_t *bnd, const uint32_t *wlen, uint32_t *slot) {
    uint32_t pos = 0, last = 0xffffffffu, acc = 0;
#pragma unroll
    for (int b = 1; b <= PACK_WARPS; b++) {
        pos += wlen[b - 1];
        const uint32_t v = bnd[b];
        bnd[b] = 0;
        if (pos & 31u) {
            const uint32_t wi = pos >> 5;
            if (wi != last) {
                if (last != 0xffffffffu) slot[last] = acc;
                last = wi;
                acc = 0;
            }
            acc |= v;
        }
    }
    if (last != 0xffffffffu) slot[last] = acc;
}

// Code tables in token-bin order (common.cuh tok_bin): code << size, and the full length per (ZRL count, bin); -> the
// ZRL (0xF0) codes of the two AC tables as code << 8 | length. The tables are k_tables' output: every load of them must
// stay behind pdl_wait() (volatile: a load through a const __restrict__ pointer may be hoisted above the wait).
__device__ __forceinline__ void pack_build_tables(PackShared &sh, const HuffDev *huff, int tid, uint32_t &zr_y, uint32_t &zr_c) {
    const volatile HuffDev *vh = huff;
    for (int i = tid; i < 1024; i += PACK_THREADS) {
        const uint32_t bin = (uint32_t)i, t = bin_table(bin), nb = (bin >> 2) & 15u;
        const bool valid = (t & 1u) || (bin >> 6) == 0u;   // DC bins carry no run
        const uint32_t sym = bin_symbol(bin);
        const uint32_t en = valid ? vh->enc[t][sym] : 0u;
        const uint32_t l = en & 0xFFu;
        sh.code[bin] = l ? ((en >> 8) << nb) : 0u;
        sh.len[bin] = (uint8_t)(l ? l + nb : 0u);
    }
    __syncthreads();
    zr_y = (sh.code[tok_bin(1, 0xF0)] << 8) | sh.len[tok_bin(1, 0xF0)];
    zr_c = (sh.code[tok_bin(3, 0xF0)] << 8) | sh.len[tok_bin(3, 0xF0)];
    for (int i = 1024 + tid; i < 4096; i += PACK_THREADS) {   // ZRL counts 1..3 (AC tokens only)
        const uint32_t bin = (uint32_t)i & 0x3FFu, nz = (uint32_t)i >> 10, l = sh.len[bin];
        const uint32_t t = bin_table(bin);
        const uint32_t zl = ((t & 2u) ? zr_c : zr_y) & 0xFFu;
        sh.len[i] = (uint8_t)((l && (t & 1u)) ? l + nz * zl : l);
    }
    __syncthreads();
}

__global__ void __launch_bounds__(PACK_THREADS, PACK_CTAS)
k_pack(const uint32_t *__restrict__ pool, const TileRec *__restrict__ recs, int ntiles, const HuffDev *huff,
       uint32_t *__restrict__ slots, uint32_t *__restrict__ tile_bits, uint32_t sub_words) {
    __shared__ __align__(16) PackShared sh;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    for (int i = tid; i < WIN_WORDS; i += PACK_THREADS) sh.buf[i] = 0;
    for (int i = tid; i < PACK_WARPS * (SUB_WORDS + 4); i += PACK_THREADS) sh.sub[0][i] = 0;
    if (tid < 2 * (PACK_WARPS + 1)) sh.bnd[0][tid] = 0;
    pdl_wait();   // everything above ran under k_tables
    uint32_t zr_y, zr_c;
    pack_build_tables(sh, huff, tid, zr_y, zr_c);
    uint32_t *sub = sh.sub[wid];

    bool pend = false;      // the previous tile's shared words are still in their cells
    uint32_t *pslot = nullptr;
    int it = 0;
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x, it++) {
        const int cur = it & 1, l3 = it % 3, pl3 = (it + 2) % 3;
        const TileRec rec = recs[t];
        // the walk starts at the 16-byte boundary below the run: virtual index v = token index + a
        const uint32_t a = rec.base & 3u;
        const uint32_t vend = a + rec.count;
        const uint4 *tk4 = reinterpret_cast<const uint4 *>(pool + (rec.base - a));
        // warp shares: contiguous, a multiple of PACK_STEP tokens; every lane owns PACK_K consecutive tokens per step
        const uint32_t per = (((vend + PACK_WARPS - 1u) / PACK_WARPS) + PACK_STEP - 1u) & ~(uint32_t)(PACK_STEP - 1);
        const uint32_t lo = min(vend, (uint32_t)wid * per), hi = min(vend, lo + per);
        // the next tile's token run on its way into L2 while this one is coded
        if (t + (int)gridDim.x < ntiles) {
            const TileRec nx = recs[t + gridDim.x];
            const char *p0 = reinterpret_cast<const char *>(pool + (nx.base & ~31u));
            const uint32_t nbytes = ((nx.base & 31u) + nx.count) * 4u;
            for (uint32_t o = tid * 128u; o < nbytes; o += PACK_THREADS * 128u)
                asm volatile("prefetch.global.L2 [%0];" ::"l"(p0 + o));
        }

        // ---- 1. code the share into the warp's buffer (or only measure it: dense tiles)
        const bool dense = rec.count > PACK_DENSE_TOKENS;
        uint32_t len;
        if (!dense) len = (uint32_t)pack_scatter<false>(sh, sub, sub_words, tk4, a, lo, hi, 0, lane, zr_y, zr_c);
        else len = pack_length(sh, tk4, a, lo, hi, lane);
        if (lane == 0) sh.wlen[l3][wid] = len;
        __syncthreads();   // ---- 2. also: every warp is done with the previous tile's cells
        if (pend && tid == 0) pack_flush_shared_words(sh.bnd[cur ^ 1], sh.wlen[pl3], pslot);
        uint32_t base = 0, total = 0;
        bool two_pass = dense;
#pragma unroll
        for (int w = 0; w < PACK_WARPS; w++) {
            const uint32_t x = sh.wlen[l3][w];
            if (w < wid) base += x;
            total += x;
            if (x > sub_words * 32u) two_pass = true;   // a warp buffer overflowed: its bits were dropped
        }
        if (tid == 0) tile_bits[t] = total;
        uint32_t *slot = slots + (size_t)t * SLOT_WORDS;

        if (!two_pass) {
            // ---- 3. shift the share into place; clear the buffer behind
            const uint32_t shv = base & 31u, fw = base >> 5;
            const uint32_t nV = (shv + len + 31u) >> 5;
            const uint32_t tailbits = (shv + len) & 31u;
            for (uint32_t i = lane; i < nV; i += 32) {
                const uint32_t hi_w = i ? sub[i - 1] : 0u, lo_w = sub[i];
                const uint32_t v = __funnelshift_r(lo_w, hi_w, shv);
                if (i == 0 && shv != 0u) atomicOr(&sh.bnd[cur][wid], v);
                else if (i == nV - 1 && tailbits != 0u) atomicOr(&sh.bnd[cur][wid + 1], v);
                else slot[fw + i] = v;
            }
            __syncwarp();
            for (uint32_t i = lane; i < nV + 1; i += 32) sub[i] = 0;
            pend = true;
            pslot = slot;
        } else {
            if (!dense) {   // overflowed buffers hold a prefix of the share: clear them
                for (uint32_t i = lane; i < (uint32_t)SUB_WORDS + 4u; i += 32) sub[i] = 0;
            }
            const uint32_t nwords = (total + 31u) >> 5;
            for (uint32_t wbase = 0; wbase < nwords; wbase += WIN_WORDS) {
                pack_scatter<true>(sh, sh.buf, WIN_WORDS, tk4, a, lo, hi, (int)base - (int)(wbase * 32u), lane, zr_y, zr_c);
                __syncthreads();
                const uint32_t wn = min((uint32_t)WIN_WORDS, nwords - wbase);
                for (uint32_t i = tid; i < wn; i += PACK_THREADS) { slot[wbase + i] = sh.buf[i]; sh.buf[i] = 0; }
                __syncthreads();
            }
            pend = false;
        }
    }
    __syncthreads();
    if (pend && tid == 0) pack_flush_shared_words(sh.bnd[(it + 1) & 1], sh.wlen[(it + 2) % 3], pslot);
}

// ------------------------------------------------------------------------------------------------------
// k_rst_pad (restart intervals, jchuff.c emit_restart): every interval but the last ends with 1-bits up to a byte
// boundary and the marker 0xFF, 0xD0 + (interval & 7). Intervals are whole MCU rows, i.e. whole tiles, and start byte
// aligned, so the padding is a function of the interval's own bit count: one thread per interval adds the bits to the
// interval's last tile (its slot has 4 spare words) before the tile scan runs. k_stuff leaves the marker's 0xFF alone.
__global__ void __launch_bounds__(128)
k_rst_pad(uint32_t *__restrict__ slots, uint32_t *__restrict__ tile_bits, int ntiles, int rst_tiles) {
    pdl_wait();
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    const long long first = (long long)j * rst_tiles, last = first + rst_tiles - 1;
    if (last >= ntiles - 1) return;   // the last interval: no marker, k_stuff pads the end of the stream
    uint64_t B = 0;
    for (long long t = first; t <= last; t++) B += tile_bits[t];
    const uint32_t pad = (8u - (uint32_t)(B & 7u)) & 7u, n = pad + 16u;
    const uint64_t v = ((uint64_t)((1u << pad) - 1u) << 16) | 0xFF00u | (0xD0u + ((uint32_t)j & 7u));
    const uint32_t tb = tile_bits[last], wi = tb >> 5, sh = tb & 31u;
    const uint64_t acc = (v << (64u - n)) >> sh;   // bits [sh, sh + n) of the two words starting at wi
    uint32_t *slot = slots + (size_t)last * SLOT_WORDS;
    slot[wi] = (sh ? (slot[wi] & ~(0xFFFFFFFFu >> sh)) : 0u) | (uint32_t)(acc >> 32);
    if (sh + n > 32u) slot[wi + 1] = (uint32_t)acc;
    tile_bits[last] = tb + n;
}

// ------------------------------------------------------------------------------------------------------
// k_scan_tiles: exclusive scan of the per-tile bit counts (ntiles ~ 4e4 for the headline image). One CTA per chunk
// of 4096 counts (16-byte coalesced loads, 4 counts per thread, warp shuffles), chunks chained by a decoupled
// look-back over `desc` (zeroed per encode; chunk ids come from a ticket so predecessors are always running).
constexpr int SCAN_CHUNK = 4096;
__global__ void __launch_bounds__(1024)
k_scan_tiles(const uint32_t *tile_bits /* k_pack's output: no __restrict__ (pdl_wait) */, int ntiles, uint64_t *__restrict__ tile_off,
             const uint32_t *__restrict__ slots, uint64_t *__restrict__ strip_bits, uint64_t *__restrict__ desc,
             uint32_t *__restrict__ ticket, uint32_t *__restrict__ chunk_tile, uint32_t nchunk_cap, uint32_t *__restrict__ err) {
    __shared__ uint32_t s_w[32];
    __shared__ uint64_t s_carry;
    __shared__ int s_chunk;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    pdl_trigger();   // k_stuff (or k_strip_seam) sets up meanwhile
    pdl_wait();
    if (tid == 0) s_chunk = (int)atomicAdd(ticket, 1u);
    __syncthreads();
    const int ch = s_chunk;
    const int i0 = ch * SCAN_CHUNK + tid * 4;
    uint32_t v[4] = {0, 0, 0, 0};
    if (i0 + 3 < ntiles) {
        const uint4 x = *reinterpret_cast<const uint4 *>(tile_bits + i0);   // tile_bits is 16-byte aligned, i0 % 4 == 0
        v[0] = x.x; v[1] = x.y; v[2] = x.z; v[3] = x.w;
    } else {
#pragma unroll
        for (int k = 0; k < 4; k++) if (i0 + k < ntiles) v[k] = tile_bits[i0 + k];
    }
    const uint32_t mine = v[0] + v[1] + v[2] + v[3];   // < 2^32: a chunk holds at most 4096 * 425984 bits
    uint32_t inc = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += y;
    }
    if (lane == 31) s_w[wid] = inc;
    __syncthreads();
    uint32_t wv = s_w[lane], winc = wv;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, winc, o);
        if (lane >= o) winc += y;
    }
    const uint32_t wbase = __shfl_sync(0xffffffffu, winc - wv, wid);
    const uint32_t ctotal = __shfl_sync(0xffffffffu, winc, 31);
    if (wid == 0) {
        const uint64_t pre = lookback_exclusive(desc, ch, ctotal, err);
        if (lane == 0) s_carry = pre;
    }
    __syncthreads();
    const uint64_t carry = s_carry;
    uint64_t run = carry + wbase + (inc - mine);
    constexpr uint64_t CHB = (uint64_t)STUFF_CHUNK * 8;   // bits per k_stuff chunk
#pragma unroll
    for (int k = 0; k < 4; k++) {
        if (i0 + k < ntiles) {
            tile_off[i0 + k] = run;
            // the k_stuff chunks whose first bit (at seam skip 0; k_stuff steps over a tile end within 7 bits) is in this tile
            for (uint64_t c = (run + CHB - 1) / CHB; c * CHB < run + v[k] && c < nchunk_cap; c++) chunk_tile[c] = (uint32_t)(i0 + k);
        }
        run += v[k];
    }
    if (ch == (int)gridDim.x - 1 && tid == 0) {
        const uint64_t T = carry + ctotal;
        tile_off[ntiles] = T;
        strip_bits[0] = T;
        strip_bits[1] = ntiles > 0 ? slots[0] : 0;
    }
}

// ------------------------------------------------------------------------------------------------------
// k_stuff: the strip's bit string (tile slots, concatenated virtually) -> shifted to the global bit phase ->
// bytes -> 0xFF00 stuffing -> final position. Persistent CTAs take chunks of unstuffed bytes in ticket order; a
// decoupled look-back over the stuffed byte
// counts gives each chunk its output offset while the other warps already stage their bytes at chunk-local offsets;
// the copy-out re-aligns to 16-byte global vectors with funnel shifts.
// Byte j of the strip = local bits [skip + 8j, skip + 8j + 8); bits past the strip's end come from `ext`
// (the next strip's first bits) followed by 1-bits (jchuff.c flush_bits padding).
constexpr int STUFF_TWIN = 72;   // tiles whose offsets are cached per chunk (a chunk of a flat image spans more)

struct StuffTiles {
    const uint64_t *s_toff;
    const uint32_t *s_tbits;
    const uint64_t *g_toff;
    const uint32_t *g_tbits;
    int tau0, ntiles;
    __device__ __forceinline__ uint64_t off(int ti) const {
        const int r = ti - tau0;
        return r < STUFF_TWIN ? s_toff[r] : g_toff[min(ti, ntiles)];
    }
    __device__ __forceinline__ uint32_t bits(int ti) const {
        const int r = ti - tau0;
        return r < STUFF_TWIN ? s_tbits[r] : g_tbits[ti];
    }
};

// 32 stream bits starting at bit p when they are not all inside one tile (tile seams, the strip's end)
__device__ __noinline__ uint32_t stuff_seam_word(const StuffTiles &tl, const uint32_t *__restrict__ slots, uint64_t &p, int &tau,
                                                 uint64_t T, int ext) {
    uint32_t res = 0;
    int got = 0;
    while (got < 32) {
        if (p >= T) {
            const uint64_t e = p - T;
            uint32_t x = 0xffffffffu;
            if (e < 32) {
                x = ((uint32_t)ext << 24) | 0x00ffffffu;
                if (e) x = (x << e) | ((1u << e) - 1u);
            }
            res |= x >> got;
            p += 32 - got;
            got = 32;
            break;
        }
        while (tl.off(tau + 1) <= p) tau++;
        const uint32_t tb = tl.bits(tau);
        const uint32_t qb = (uint32_t)(p - tl.off(tau));
        const uint32_t rem = tb - qb;
        const uint32_t *slot = slots + (size_t)tau * SLOT_WORDS;
        const uint32_t wi = qb >> 5, sh = qb & 31u;
        const uint32_t nw = (tb + 31u) >> 5;
        const uint32_t w0 = slot[wi];
        const uint32_t w1 = (sh && wi + 1 < nw) ? slot[wi + 1] : 0u;
        uint32_t x = sh ? ((w0 << sh) | (w1 >> (32 - sh))) : w0;
        const int take = min(32 - got, (int)min(rem, 32u));
        if (take < 32) x &= ~(0xffffffffu >> take);
        res |= x >> got;
        got += take;
        p += take;
    }
    return res;
}

// One 32-bit piece of the stream (w: first byte in bits 31..24) -> its bytes in memory order with a 0x00 after every
// 0xFF, OR-ed into the zeroed staging buffer at byte offset o (any alignment). Branch-free: the byte expansion is two
// PRMTs whose selectors come from a 16-entry table indexed by the word's 0xFF mask. Returns the bytes produced.
// `keep`: 0x01 in byte b (memory order) unless byte b is the 0xFF of a restart marker, which takes no 0x00.
__device__ __forceinline__ uint32_t stuff_place_word(uint32_t w, uint32_t o, uint32_t sbase, const uint32_t *s_lut,
                                                     uint32_t keep = 0x01010101u) {
    const uint32_t l = __byte_perm(w, 0, 0x0123);
    uint32_t mm = l & (l >> 4) & 0x0F0F0F0Fu;   // a byte is 0xFF iff all eight bits survive the and-fold
    mm &= mm >> 2;
    mm &= mm >> 1;
    mm &= keep;
    const uint32_t m4 = (mm * 0x01020408u) >> 24;   // bit i: byte i is 0xFF
    const uint32_t sel = s_lut[m4];
    const uint32_t lo = __byte_perm(l, 0, sel & 0xFFFFu), hi = __byte_perm(l, 0, sel >> 16);
    const uint32_t bs = (o & 3u) * 8u;
    const uint32_t addr = sbase + (o & ~3u);
    const uint32_t x0 = lo << bs, x1 = __funnelshift_l(lo, hi, bs), x2 = __funnelshift_l(hi, 0u, bs);
    asm volatile("red.shared.or.b32 [%0], %1;" ::"r"(addr), "r"(x0) : "memory");
    asm volatile("red.shared.or.b32 [%0+4], %1;" ::"r"(addr), "r"(x1) : "memory");
    if (x2) asm volatile("red.shared.or.b32 [%0+8], %1;" ::"r"(addr), "r"(x2) : "memory");
    return 4u + __popc(m4);
}

template <bool RST>
__global__ void __launch_bounds__(STUFF_THREADS, STUFF_CTAS)
k_stuff(StuffArgs a) {
    constexpr int NWARP = STUFF_THREADS / 32;
    constexpr int NP = STUFF_PIECES;                       // 16-byte pieces per thread and chunk
    constexpr int PSTRIDE = STUFF_THREADS * 16;            // bytes between a thread's pieces
    constexpr int OUT_WORDS = (2 * STUFF_CHUNK + 64) / 4;
    __shared__ uint64_t s_toff[STUFF_TWIN];
    __shared__ uint32_t s_tbits[STUFF_TWIN];
    __shared__ int s_chunk;
    __shared__ uint32_t s_warp[NP][NWARP];
    __shared__ uint64_t s_goff;
    __shared__ uint32_t s_lut[16];
    __shared__ __align__(16) uint32_t s_out32[OUT_WORDS];
    uint8_t *s_out = reinterpret_cast<uint8_t *>(s_out32);
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const uint32_t sbase = smem_u32(s_out32);

    if (tid < 16) {   // PRMT selectors: bytes 0..3 of the word in order, a zero byte (selector 4) after every 0xFF
        uint32_t sel = 0;
        int n = 0;
        for (int i = 0; i < 4; i++) {
            sel |= (uint32_t)i << (4 * n++);
            if (tid & (1 << i)) sel |= 4u << (4 * n++);
        }
        for (; n < 8; n++) sel |= 4u << (4 * n);
        s_lut[tid] = sel;
    }
    for (int i = tid; i < OUT_WORDS; i += STUFF_THREADS) s_out32[i] = 0;
    pdl_wait();   // the set-up above ran under the tile scan
    const uint64_t T = a.tile_off[a.ntiles];
    const int a_skip = a.seam[0], a_ext = a.seam[1] ^ 0xFF;   // the ext byte is stored inverted: zeroed control block = whole image
    const uint64_t NB = T > (uint64_t)a_skip ? (T - a_skip + 7) >> 3 : 0;
    const int nchunks = (int)max((uint64_t)1, (NB + STUFF_CHUNK - 1) / STUFF_CHUNK);
    const uint32_t hdr = a.huff->hdr_len;

    for (;;) {
        // chunk ids are taken when the work starts (a ticket held back would make its successors spin in the look-back)
        if (tid == 0) s_chunk = (int)atomicAdd(a.ticket, 1u);
        __syncthreads();
        const int ch = s_chunk;
        if (ch >= nchunks) break;
        const uint64_t j0c = (uint64_t)ch * STUFF_CHUNK;
        const uint64_t p0c = (uint64_t)a_skip + 8 * j0c;
        // tile holding the chunk's first bit: the tile scan left it in chunk_tile (for skip 0; with a seam skip the first
        // bit may lie up to 7 bits further, i.e. in the next tile: the pieces' own tile walk steps over that)
        const int tau0 = (int)a.chunk_tile[ch];
        for (int i = tid; i < STUFF_TWIN; i += STUFF_THREADS) {
            const int ti = min(tau0 + i, a.ntiles);
            s_toff[i] = a.tile_off[ti];
            s_tbits[i] = ti < a.ntiles ? a.tile_bits[ti] : 0;
        }
        __syncthreads();
        StuffTiles tl{s_toff, s_tbits, a.tile_off, a.tile_bits, tau0, a.ntiles};

        // ---- NP pieces of 16 bytes per thread: w[i][q] = stream bits [p + 32q, p + 32q + 32) of piece i, MSB first
        uint32_t w[NP][4];
        int nvalid[NP];
        uint32_t cnt[NP];
        uint32_t marker[NP];   // RST: bit k set = byte k of the piece is a restart marker's 0xFF (not stuffed)
        int tau = tau0;
#pragma unroll
        for (int i = 0; i < NP; i++) {
            const uint64_t jb = j0c + (uint64_t)i * PSTRIDE + (uint64_t)tid * 16;
            nvalid[i] = jb >= NB ? 0 : (int)min((uint64_t)16, NB - jb);
#pragma unroll
            for (int q = 0; q < 4; q++) w[i][q] = 0;
            marker[i] = 0;
            if (nvalid[i] > 0) {
                uint64_t p = (uint64_t)a_skip + 8 * jb;
                while (tl.off(tau + 1) <= p) tau++;
                uint64_t tstart = tl.off(tau), tend = tl.off(tau + 1);
                if (RST) {   // the markers inside this piece: the one that ends the interval of its first bit, and (tiny
                             // intervals) the ones that follow while they still begin inside the piece
                    int iv_last = (tau / a.rst_tiles + 1) * a.rst_tiles - 1;
                    while (iv_last < a.ntiles - 1) {
                        const long long m = (long long)(tl.off(iv_last + 1) >> 3) - 2 - (long long)jb;
                        if (m >= 16) break;
                        if (m >= 0) marker[i] |= 1u << m;
                        iv_last += a.rst_tiles;
                    }
                }
                if (p + 128 <= tend) {  // all bits inside one tile
                    const uint32_t qb = (uint32_t)(p - tstart);
                    const uint32_t *slot = a.slots + (size_t)tau * SLOT_WORDS + (qb >> 5);
                    const uint32_t sh = qb & 31u;
                    uint32_t x[5];
#pragma unroll
                    for (int q = 0; q < 5; q++) x[q] = slot[q];   // slot[4] may belong to the next tile: shifted out when sh == 0
#pragma unroll
                    for (int q = 0; q < 4; q++) w[i][q] = __funnelshift_l(x[q + 1], x[q], sh);
                } else {                // a tile seam (or the strip's end) inside these 16 bytes: word by word
#pragma unroll
                    for (int q = 0; q < 4; q++) {
                        if (p + 32 <= tend) {
                            const uint32_t qb = (uint32_t)(p - tstart);
                            const uint32_t *slot = a.slots + (size_t)tau * SLOT_WORDS + (qb >> 5);
                            w[i][q] = __funnelshift_l(slot[1], slot[0], qb & 31u);
                            p += 32;
                        } else {
                            w[i][q] = stuff_seam_word(tl, a.slots, p, tau, T, a_ext);
                            if (p < T) {
                                while (tl.off(tau + 1) <= p) tau++;
                                tstart = tl.off(tau);
                                tend = tl.off(tau + 1);
                            } else {
                                tend = 0;   // past the strip's end: stay on the seam path
                            }
                        }
                    }
                }
            }
            // stuffed size of the piece
            int nff = 0;
#pragma unroll
            for (int q = 0; q < 4; q++) {
                uint32_t m = w[i][q] & (w[i][q] >> 4) & 0x0F0F0F0Fu;
                m &= m >> 2;
                m &= m >> 1;
                m &= 0x01010101u;
                if (nvalid[i] < 16) {  // tail piece: ignore bytes past the end
#pragma unroll
                    for (int bb = 0; bb < 4; bb++)
                        if (4 * q + bb >= nvalid[i]) m &= ~(1u << (24 - 8 * bb));
                }
                if (RST) {
#pragma unroll
                    for (int bb = 0; bb < 4; bb++)
                        if ((marker[i] >> (4 * q + bb)) & 1u) m &= ~(1u << (24 - 8 * bb));
                }
                nff += __popc(m);
            }
            cnt[i] = (uint32_t)(nvalid[i] + nff);
        }
        // ---- offsets: bytes are ordered piece-major (piece i of all threads, then piece i + 1)
        uint32_t inc[NP];
#pragma unroll
        for (int i = 0; i < NP; i++) inc[i] = cnt[i];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
#pragma unroll
            for (int i = 0; i < NP; i++) {
                const uint32_t y = __shfl_up_sync(0xffffffffu, inc[i], o);
                if (lane >= o) inc[i] += y;
            }
        }
        if (lane == 31) {
#pragma unroll
            for (int i = 0; i < NP; i++) s_warp[i][wid] = inc[i];
        }
        __syncthreads();
        uint32_t off[NP], total = 0;
#pragma unroll
        for (int i = 0; i < NP; i++) {
            uint32_t wb = 0, tt = 0;
#pragma unroll
            for (int k = 0; k < NWARP; k++) {
                const uint32_t x = s_warp[i][k];
                if (k < wid) wb += x;
                tt += x;
            }
            off[i] = total + wb + inc[i] - cnt[i];
            total += tt;
        }
        if (wid == 0) {   // the other warps stage their bytes meanwhile
            const uint64_t pre = lookback_exclusive(a.desc, ch, total, a.err);
            if (lane == 0) s_goff = pre;
        }
        // ---- stage the stuffed bytes at their chunk-local offsets (the buffer is all zero here)
#pragma unroll
        for (int i = 0; i < NP; i++) {
            uint32_t o = off[i];
            if (nvalid[i] == 16) {
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    uint32_t keep = 0x01010101u;
                    if (RST) {
                        const uint32_t mk = (marker[i] >> (4 * q)) & 15u;   // bit bb: byte bb of this word (memory order)
                        keep &= ~((mk & 1u) | ((mk & 2u) << 7) | ((mk & 4u) << 14) | ((mk & 8u) << 21));
                    }
                    o += stuff_place_word(w[i][q], o, sbase, s_lut, keep);
                }
            } else {
                for (int k = 0; k < nvalid[i]; k++) {
                    uint32_t byte = 0;
#pragma unroll
                    for (int q = 0; q < 4; q++) if ((k >> 2) == q) byte = (w[i][q] >> (24 - 8 * (k & 3))) & 0xFFu;
                    atomicOr(&s_out32[o >> 2], byte << ((o & 3u) * 8u));
                    o += (byte == 0xFFu && !(RST && ((marker[i] >> k) & 1u))) ? 2u : 1u;
                }
            }
        }
        __syncthreads();
        // ---- copy out: 16-byte aligned global vectors assembled from the (unaligned) staged bytes
        const uint64_t goff = (uint64_t)hdr + s_goff;
        const bool last = ch == nchunks - 1;
        const uint64_t end = goff + total + ((last && a.append_eoi) ? 2 : 0);
        if (end > a.cap) {
            if (tid == 0) *a.err = 3;
        } else {
            uint8_t *dst = a.out + goff;                     // byte k of the chunk -> dst[k]
            const uint32_t mis = (uint32_t)(reinterpret_cast<uintptr_t>(dst) & 15u);
            // vector v covers chunk bytes [16 v - mis, 16 v - mis + 16)
            for (uint32_t v = tid; 16 * v < total + mis; v += STUFF_THREADS) {
                const int k0 = (int)(16 * v) - (int)mis;
                if (k0 >= 0 && (uint32_t)k0 + 16 <= total) {
                    const uint32_t wi = (uint32_t)k0 >> 2, bs = ((uint32_t)k0 & 3u) * 8u;
                    const uint32_t x0 = s_out32[wi], x1 = s_out32[wi + 1], x2 = s_out32[wi + 2], x3 = s_out32[wi + 3], x4 = s_out32[wi + 4];
                    uint4 o4;
                    o4.x = __funnelshift_r(x0, x1, bs); o4.y = __funnelshift_r(x1, x2, bs);
                    o4.z = __funnelshift_r(x2, x3, bs); o4.w = __funnelshift_r(x3, x4, bs);
                    *reinterpret_cast<uint4 *>(dst + k0) = o4;
                } else {
                    for (int k = max(k0, 0); k < min(k0 + 16, (int)total); k++) dst[k] = s_out[k];
                }
            }
            if (last && a.append_eoi && tid == 0) { a.out[goff + total] = 0xFF; a.out[goff + total + 1] = 0xD9; }
        }
        if (last && tid == 0) *a.out_len = end;
        __syncthreads();
        // clear what was staged (the last stuffed byte may carry its 0x00 one byte further)
        for (uint32_t i = tid; i * 16 < total + 20; i += STUFF_THREADS) reinterpret_cast<uint4 *>(s_out32)[i] = make_uint4(0, 0, 0, 0);
    }
}

// ------------------------------------------------------------------------------------------------------
cudaError_t launch_tables(const uint32_t *hist, int optimize, HuffDev *huff, const QuantDev *qd, int full_w, int full_h,
                          int hs, int vs, int nc, uint8_t *out, int emit_header, int restart_interval, uint32_t *err_out, cudaStream_t s) {
    if (nc == 1)
        return launch_pdl(k_tables<1>, dim3(1), dim3(128), 0, s, hist, optimize, huff, qd, full_w, full_h, hs, vs, out, emit_header, restart_interval, err_out);
    return launch_pdl(k_tables<3>, dim3(1), dim3(128), 0, s, hist, optimize, huff, qd, full_w, full_h, hs, vs, out, emit_header, restart_interval, err_out);
}
cudaError_t launch_pack(const uint32_t *pool, const TileRec *recs, const Geom &g, const HuffDev *huff,
                        uint32_t *slots, uint32_t *tile_bits, int small_buffers, cudaStream_t s) {
    const int grid = min(g.ntiles, 148 * PACK_CTAS);
    return launch_pdl(k_pack, dim3(grid), dim3(PACK_THREADS), 0, s, pool, recs, g.ntiles, huff, slots, tile_bits, small_buffers ? 24u : (uint32_t)SUB_WORDS);
}
cudaError_t launch_rst_pad(uint32_t *slots, uint32_t *tile_bits, int ntiles, int rst_tiles, cudaStream_t s) {
    const int nint = (ntiles + rst_tiles - 1) / rst_tiles;
    return launch_pdl(k_rst_pad, dim3((nint + 127) / 128), dim3(128), 0, s, slots, tile_bits, ntiles, rst_tiles);
}
int scan_desc_count(int ntiles) { return (ntiles + SCAN_CHUNK - 1) / SCAN_CHUNK + 1; }
cudaError_t launch_scan_tiles(const uint32_t *tile_bits, int ntiles, uint64_t *tile_off, const uint32_t *slots,
                              uint64_t *strip_bits, uint64_t *desc, uint32_t *ticket, uint32_t *chunk_tile, uint32_t nchunk_cap,
                              uint32_t *err, cudaStream_t s) {
    const int grid = max(1, (ntiles + SCAN_CHUNK - 1) / SCAN_CHUNK);
    return launch_pdl(k_scan_tiles, dim3(grid), dim3(1024), 0, s, tile_bits, ntiles, tile_off, slots, strip_bits, desc, ticket, chunk_tile, nchunk_cap, err);
}
__global__ void k_set_seam(int *seam, int skip, int ext) { seam[0] = skip; seam[1] = ext ^ 0xFF; }

// bits_all[k] = {entropy bits of strip k, its first 32 bits (top-aligned)}: strip `rank` starts at global bit G =
// sum of the bit counts before it; it skips the (8 - G % 8) % 8 bits that complete the previous strip's last byte and
// borrows the next strip's first byte for its own last one (1-bits after the last strip).
__global__ void k_seam_from_bits(int *seam, const int64_t *__restrict__ bits_all, int rank, int world) {
    uint64_t G = 0;
    for (int k = 0; k < rank; k++) G += (uint64_t)bits_all[2 * k];
    seam[0] = (int)((8u - (uint32_t)(G & 7u)) & 7u);
    seam[1] = (rank == world - 1 ? 0xFF : (int)(((uint64_t)bits_all[2 * (rank + 1) + 1] >> 24) & 0xFFu)) ^ 0xFF;
}

// ---- one-collective strip exchange -------------------------------------------------------------------------
// After the all-gather of every strip's StripRecord each rank has what the three-collective schedule exchanged:
// the image histogram is the sum of the strips' plus the DC symbols at the strip starts (derived from first_dc /
// last_dc of neighbouring records); a strip's entropy bit count is its histogram weighted with the code lengths,
// so the bit phase of every strip is known without waiting for the others' entropy coders; the byte completing a
// strip's last byte is the head of the next strip's record tokens coded with the (identical) tables.
__device__ __forceinline__ uint32_t dc_token(int c, int diff) {
    const int nb = 32 - __clz(diff < 0 ? -diff : diff);
    return tok_dc(c ? 2u : 0u, (uint32_t)nb, (uint32_t)(diff + (diff >> 31)) & ((1u << nb) - 1u));
}

__device__ __forceinline__ uint32_t ld_acquire_sys_u32(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// Peer exchange, sending side: CTA p stores this strip's record into rank p's arena (its own included) and raises
// the flag there. The flag store follows a system-scope fence that follows every data store of the CTA.
__global__ void __launch_bounds__(256)
k_strip_push(const StripRecord *__restrict__ mine, XchgArena *const *__restrict__ peers, int rank, uint32_t seq) {
    pdl_trigger();
    pdl_wait();
    XchgArena *dst = peers[blockIdx.x];
    const int set = (int)(seq % XCHG_SETS);
    const uint4 *src = reinterpret_cast<const uint4 *>(mine);
    uint4 *d4 = reinterpret_cast<uint4 *>(&dst->rec[set][rank]);
    for (int i = threadIdx.x; i < (int)(sizeof(StripRecord) / 16); i += 256) d4[i] = src[i];
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(&dst->flags[set][rank]), "r"(seq) : "memory");
}

__global__ void __launch_bounds__(1024)
k_strip_merge(const StripRecord *rec, int rank, int world, uint32_t *__restrict__ hist,
              uint32_t *__restrict__ pool, const TileRec *__restrict__ recs, const uint32_t *flags, uint32_t seq,
              unsigned long long timeout_ns, uint32_t *__restrict__ err) {
    const int tid = threadIdx.x;
    pdl_trigger();
    pdl_wait();
    if (flags) {   // peer exchange: the records of image `seq` arrive from the other GPUs (bounded wait, never a hang)
        if (tid < world) {
            unsigned long long t0, t1;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
            while (ld_acquire_sys_u32(flags + tid) != seq) {
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
                if (t1 - t0 > timeout_ns) { atomicMax(err, 9u); break; }
                __nanosleep(100);
            }
        }
        __syncthreads();
    }
    for (int i = tid; i < 4 * 257; i += 1024) {
        uint32_t s = 0;
        for (int k = 0; k < world; k++) s += rec[k].hist[i];
        hist[i] = s;
    }
    __syncthreads();
    if (tid < world * 3) {
        const int k = tid / 3, c = tid - k * 3;
        const int diff = (int)rec[k].first_dc[c] - (k ? (int)rec[k - 1].last_dc[c] : 0);
        const uint32_t tk = dc_token(c, diff);
        atomicAdd(&hist[(c ? 2 : 0) * 257 + ((tk >> 18) & 15u)], 1u);
        if (k == rank) {   // this strip's own first MCU: the raw-DC tokens k_dc_edge_hist left alone
            const TileRec r = recs[0];
            pool[r.base + (c == 0 ? 0u : (c == 1 ? r.pos_cb : r.pos_cr))] = tk;
        }
    }
}

// seam[] of strip `rank` from the gathered records and the final code tables; also checks the strip's predicted bit
// count against what its entropy coder produced (strip_bits[0]).
__global__ void __launch_bounds__(1024)
k_strip_seam(const StripRecord *__restrict__ rec, int rank, int world, HuffDev *__restrict__ huff, int drop_header,
             int *__restrict__ seam, const uint64_t *__restrict__ strip_bits, uint32_t *__restrict__ err) {
    __shared__ unsigned long long s_red[2][32];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int t = tid >> 8, sym = tid & 255;
    pdl_trigger();   // k_stuff sets up meanwhile
    pdl_wait();
    const uint32_t len = huff->enc[t][sym] & 0xFFu;
    const uint32_t cost = len + ((t & 1) ? (uint32_t)(sym & 15) : (uint32_t)sym);
    unsigned long long before = 0, own = rec[rank].hist[t * 257 + sym];
    for (int k = 0; k < rank; k++) before += rec[k].hist[t * 257 + sym];
    uint32_t bad = (before + own) && !len;   // a counted symbol without a code
    before *= cost; own *= cost;
    if (tid <= rank * 3 + 2) {               // DC symbols at the strip starts 0..rank
        const int k = tid / 3, c = tid - k * 3;
        const uint32_t tk = dc_token(c, (int)rec[k].first_dc[c] - (k ? (int)rec[k - 1].last_dc[c] : 0));
        const uint32_t nb = (tk >> 18) & 15u, l = huff->enc[c ? 2 : 0][nb] & 0xFFu;
        bad |= !l;
        if (k < rank) before += l + nb; else own += l + nb;
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        before += __shfl_xor_sync(0xffffffffu, before, o);
        own += __shfl_xor_sync(0xffffffffu, own, o);
        bad |= __shfl_xor_sync(0xffffffffu, bad, o);
    }
    if (lane == 0) { s_red[0][wid] = before; s_red[1][wid] = own | ((unsigned long long)bad << 63); }
    __syncthreads();
    if (tid) return;
    before = own = 0;
    for (int w = 0; w < 32; w++) { before += s_red[0][w]; own += s_red[1][w] & ~(1ull << 63); bad |= (uint32_t)(s_red[1][w] >> 63); }
    seam[0] = (int)((8u - (uint32_t)(before & 7u)) & 7u);
    uint32_t ext = 0xFF;
    if (rank + 1 < world) {   // head of the next strip's bit string
        const StripRecord &nx = rec[rank + 1];
        uint64_t acc = 0; int n = 0;
        for (uint32_t j = 0; j < nx.ntok && n < 8; j++) {
            uint32_t tk = nx.tok[j];
            if (tk & TOK_RAWDC) {
                const int c = (tk >> 18) & 3u;
                tk = dc_token(c, (int)(int16_t)(tk & 0xFFFFu) - (int)rec[rank].last_dc[c]);
            }
            const uint32_t bin = (tk >> 16) & 0x3FFu, tb = bin_table(bin), nv = (bin >> 2) & 15u;
            const uint32_t sy = bin_symbol(bin);
            const uint32_t zr = huff->enc[tb][0xF0];
            for (uint32_t z = 0; z < ((tk >> 26) & 3u); z++) { acc = (acc << (zr & 0xFFu)) | (zr >> 8); n += zr & 0xFFu; }
            const uint32_t en = huff->enc[tb][sy];
            acc = (acc << (en & 0xFFu)) | (en >> 8); n += en & 0xFFu;
            acc = (acc << nv) | (tk & 0xFFFFu); n += nv;
            bad |= !(en & 0xFFu);
        }
        if (n < 8) { bad = 1; n = 8; }   // a strip shorter than one byte cannot supply the seam
        ext = (uint32_t)(acc >> (n - 8)) & 0xFFu;
    }
    seam[1] = (int)(ext ^ 0xFFu);
    if (drop_header) huff->hdr_len = 0;   // only the first strip's output starts with SOI..SOS
    if (bad || own != strip_bits[0]) atomicMax(err, 7u);
}

cudaError_t launch_strip_merge(const StripRecord *rec, int rank, int world, uint32_t *hist, uint32_t *pool,
                               const TileRec *recs, const uint32_t *flags, uint32_t seq, unsigned long long timeout_ns,
                               uint32_t *err, cudaStream_t s) {
    return launch_pdl(k_strip_merge, dim3(1), dim3(1024), 0, s, rec, rank, world, hist, pool, recs, flags, seq, timeout_ns, err);
}
cudaError_t launch_strip_push(const StripRecord *mine, XchgArena *const *peers, int rank, int world, uint32_t seq, cudaStream_t s) {
    return launch_pdl(k_strip_push, dim3(world), dim3(256), 0, s, mine, peers, rank, seq);
}
cudaError_t launch_strip_seam(const StripRecord *rec, int rank, int world, HuffDev *huff, int drop_header, int *seam,
                              const uint64_t *strip_bits, uint32_t *err, cudaStream_t s) {
    return launch_pdl(k_strip_seam, dim3(1), dim3(1024), 0, s, rec, rank, world, huff, drop_header, seam, strip_bits, err);
}

cudaError_t launch_set_seam(int *seam, int skip, int ext, cudaStream_t s) {
    k_set_seam<<<1, 1, 0, s>>>(seam, skip, ext);
    return cudaGetLastError();
}
cudaError_t launch_seam_from_bits(int *seam, const int64_t *bits_all, int rank, int world, cudaStream_t s) {
    k_seam_from_bits<<<1, 1, 0, s>>>(seam, bits_all, rank, world);
    return cudaGetLastError();
}

cudaError_t launch_stuff(const StuffArgs &a, int grid, cudaStream_t s) {
    return a.rst_tiles ? launch_pdl(k_stuff<true>, dim3(grid), dim3(STUFF_THREADS), 0, s, a)
                       : launch_pdl(k_stuff<false>, dim3(grid), dim3(STUFF_THREADS), 0, s, a);
}

}  // namespace b2j
