// dec_prog.cu -- progressive (SOF2) decode: what the reference as shipped writes (NVJPEG_ENCODING_PROGRESSIVE_DCT_HUFFMAN,
// ImageCompressorImpl.cu:28) and nvJPEG's decoder accepts (:361-366). Every scan is absorbed into the coefficient
// array in file order (jdphuff.c decode_mcu_DC_first / DC_refine / AC_first / AC_refine; tests compare the pixels with
// the CPU checker and cv2.imdecode), then the baseline back end runs (k_idct on the coefficients' own DCs, k_upcolor).
//
// A scan is one sequential Huffman chain per restart interval, and a refinement scan cannot be cut into guessed
// subsequences at all: how many correction bits a block consumes depends on which of its coefficients are already
// non-zero, i.e. on the block index. What CAN be taken off the chain is everything that is not symbol parsing:
//   * k_destuff<true> (the baseline decoder's kernel) removes the stuffing and the RSTn markers of the scan in parallel
//     and records where every interval begins, so the chain reads plain words;
//   * the non-zero history of every block is kept as a 64-bit mask (one bit per zig-zag position). A refinement scan
//     gathers the masks of its component in scan order (k_prog_gather), the chain (k_prog_scan) then only PARSES: for
//     every Huffman symbol it finds the target position and the number of correction bits with bit operations on the
//     mask (select the r-th zero, popcount) and reads them in one go; a block inside an EOB run costs one popcount.
//     It writes three words per block (correction bits, new positions, their signs) and never touches a coefficient;
//   * k_prog_apply applies those words to the coefficients, one thread per block, in parallel.
// First scans (DC, AC) write their coefficients with posted stores and OR the new positions into the masks.
// One thread per restart interval runs the chain; a file without restart markers has one interval per scan.
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "common.cuh"
#include "dec.h"
#include "dec_kernels.h"

namespace b2j {

struct ProgTable {                       // one Huffman table (dec_parse.cpp huff_derive)
    uint16_t lut[1 << PROG_LUT_BITS];    // (len << 8) | symbol for codes of length <= PROG_LUT_BITS, else 0
    int32_t maxcode[18];
    int32_t valoff[17];
    uint8_t vals[256];
};
struct ProgScanDev {
    ProgTable tb[2][3];                  // [0 DC | 1 AC][component of the scan]
    int ncomp, comp[3], Ss, Se, Ah, Al, ri;
    uint32_t nint_max;                   // restart intervals the scan can have
    uint64_t units;                      // MCUs (interleaved) or blocks of the component
};
struct ProgCtl {                         // device words of one scan's front end
    uint64_t u_len, avail;
    uint32_t ticket, nmark, err, pad;
};

// streaming bit reader over UNSTUFFED bytes: the next `nav` bits left-aligned in acc; words come from a four-word
// register queue refilled with 16-byte loads issued one vector ahead (the load latency stays off the symbol chain).
// Bytes at and after `end` (the end of the interval's data) read as zeros, as jdhuff.c jpeg_fill_bit_buffer feeds
// zero bits at a marker; over() tells that a bit past the end has been consumed (libjpeg's insufficient_data).
struct WordReader {
    const uint4 *u4;
    uint64_t acc;
    int nav, qn;
    uint32_t w0, w1, w2, w3;
    uint4 ahead;
    size_t vidx;
    int64_t wpos, end;   // byte offset of the next word into acc; end of the data (-1: an interval the file lacks)
    __device__ __forceinline__ uint32_t next_word() {
        if (qn == 0) {
            w0 = ahead.x; w1 = ahead.y; w2 = ahead.z; w3 = ahead.w;
            qn = 4;
            vidx++;
            ahead = u4[vidx];
        }
        const uint32_t w = __byte_perm(w0, 0, 0x0123);
        w0 = w1; w1 = w2; w2 = w3;
        qn--;
        const int64_t rem = end - wpos;
        wpos += 4;
        if (rem >= 4) return w;
        return rem <= 0 ? 0u : w & ~(0xFFFFFFFFu >> (8 * (int)rem));
    }
    __device__ __forceinline__ bool over() const { return wpos * 8 - nav > end * 8; }
    __device__ __forceinline__ void seek(const uint8_t *u, uint64_t byte_pos, int64_t end_pos) {   // interval starts are byte aligned
        end = end_pos;
        wpos = (int64_t)(byte_pos & ~(uint64_t)3);
        u4 = reinterpret_cast<const uint4 *>(u);
        const size_t widx = (size_t)(byte_pos >> 2);
        vidx = widx >> 2;
        const uint4 cur = u4[vidx];
        w0 = cur.x; w1 = cur.y; w2 = cur.z; w3 = cur.w;
        qn = 4;
        vidx++;
        ahead = u4[vidx];
        for (int i = 0; i < (int)(widx & 3); i++) { w0 = w1; w1 = w2; w2 = w3; qn--; }
        const uint32_t a = next_word(), b = next_word();
        const int sh = (int)(byte_pos & 3) * 8;
        acc = (((uint64_t)a << 32) | b) << sh;
        nav = 64 - sh;
    }
    __device__ __forceinline__ void fill() {
        if (nav <= 32) {
            acc |= (uint64_t)next_word() << (32 - nav);
            nav += 32;
        }
    }
    __device__ __forceinline__ uint32_t get(int n) {   // 0 <= n <= 32
        if (n == 0) return 0;
        fill();
        const uint32_t v = (uint32_t)(acc >> (64 - n));
        acc <<= n;
        nav -= n;
        return v;
    }
    __device__ __forceinline__ uint64_t get64(int n) {   // 0 <= n <= 63
        if (n <= 32) return get(n);
        const uint64_t hi = get(n - 32);
        return (hi << 32) | get(32);
    }
    __device__ __forceinline__ int sym(const ProgTable &t) {
        fill();
        const uint32_t top = (uint32_t)(acc >> 48);
        const uint32_t e = t.lut[top >> (16 - PROG_LUT_BITS)];
        int l = 16, s = 0;   // invalid code: jdhuff.c warns and returns 0
        if (e) { l = (int)(e >> 8); s = (int)(e & 0xFF); }
        else
            for (int q = PROG_LUT_BITS + 1; q <= 16; q++) {
                const int code = (int)(top >> (16 - q));
                if (code <= t.maxcode[q]) { l = q; s = t.vals[(t.valoff[q] + code) & 255]; break; }
            }
        acc <<= l;
        nav -= l;
        return s;
    }
};

__device__ __forceinline__ int prog_extend(int v, int n) { return n == 0 ? 0 : (v < (1 << (n - 1)) ? v - (1 << n) + 1 : v); }

// scan-order index of block (bx, by) of component c (jdcoefct.c: non-interleaved scans walk the component's own blocks)
__host__ __device__ __forceinline__ size_t prog_block_index(const Geom &g, int c, int bx, int by) {
    const int h = c ? 1 : g.hs, v = c ? 1 : g.vs;
    const int mx = bx / h, my = by / v;
    const int blkn = c ? g.bpm - 3 + c : (by % v) * h + (bx % h);
    return ((size_t)my * g.mcux + mx) * g.bpm + blkn;
}
__device__ __forceinline__ size_t prog_unit_block(const Geom &g, int c, uint64_t u) {
    const int wib = g.wib[c];
    return prog_block_index(g, c, (int)(u % wib), (int)(u / wib));
}

// the blocks of one component in scan (raster) order without a division per block: the chain's per-block overhead
struct UnitWalk {
    int bx, by, wib, c;
    __device__ __forceinline__ void init(const Geom &g, int comp, uint64_t u) { c = comp; wib = g.wib[comp]; by = (int)(u / (uint64_t)wib); bx = (int)(u - (uint64_t)by * wib); }
    __device__ __forceinline__ size_t block(const Geom &g) const {
        if (c) return ((size_t)by * g.mcux + bx) * g.bpm + (g.bpm - 3 + c);
        const int mx = bx / g.hs, my = by / g.vs;   // hs, vs in {1, 2, 4}: shifts after inlining would need them constant; small ints
        return ((size_t)my * g.mcux + mx) * g.bpm + (by - my * g.vs) * g.hs + (bx - mx * g.hs);
    }
    __device__ __forceinline__ void next() { if (++bx == wib) { bx = 0; by++; } }
};

__device__ __forceinline__ uint64_t bits_range(int lo, int hi) {   // bits lo..hi inclusive (0 <= lo, hi <= 63), empty if lo > hi
    if (lo > hi) return 0;
    return (~0ull >> (63 - hi)) & (~0ull << lo);
}
// position of the (r + 1)-th set bit of z (r >= 0), or 64 if z has at most r set bits
__device__ __forceinline__ int select_bit(uint64_t z, int r) {
    const uint32_t lo = (uint32_t)z, hi = (uint32_t)(z >> 32);
    const int nlo = __popc(lo);
    if (r < nlo) return (int)__fns(lo, 0, r + 1);
    r -= nlo;
    if (r < __popc(hi)) return 32 + (int)__fns(hi, 0, r + 1);
    return 64;
}

// refinement scans: the non-zero history of the scan's component in scan order
__global__ void __launch_bounds__(256)
k_prog_gather(const uint64_t *__restrict__ mask, uint64_t *__restrict__ cm, Geom g, int c, uint64_t units) {
    const uint64_t u = (uint64_t)blockIdx.x * 256 + threadIdx.x;
    if (u < units) cm[u] = mask[prog_unit_block(g, c, u)];
}

// the chain: one thread per restart interval. bnd[j] = byte offset (unstuffed) where interval j + 1 begins.
__global__ void __launch_bounds__(32)
k_prog_scan(const uint8_t *__restrict__ u, const ProgCtl *__restrict__ ctl, const uint32_t *__restrict__ bnd,
            const ProgScanDev *__restrict__ scd, Geom g, int16_t *__restrict__ coef, uint64_t *__restrict__ mask,
            const uint64_t *__restrict__ cm, uint64_t *__restrict__ corr, uint64_t *__restrict__ newm, uint64_t *__restrict__ news) {
    __shared__ ProgScanDev sc;
    {
        const uint32_t *src = reinterpret_cast<const uint32_t *>(scd);
        uint32_t *dst = reinterpret_cast<uint32_t *>(&sc);
        for (int i = threadIdx.x; i < (int)(sizeof(ProgScanDev) / 4); i += 32) dst[i] = src[i];
    }
    __syncwarp();
    const uint32_t j = blockIdx.x * 32 + threadIdx.x;
    const uint32_t nint = sc.ri ? ctl->nmark + 1u : 1u;
    // Interval j ends where the next begins, the last one where the data ends. A cut file lacks the intervals from
    // nint on: they read as out of data from their start, so they leave their blocks alone (jdphuff.c insufficient_data)
    // and a refinement scan writes zero words for them. Interval nint is the previous thread's: when the data ends
    // exactly at its start, libjpeg still decodes one MCU of zero bits there.
    if (j >= sc.nint_max || j == nint) return;
    WordReader r;
    if (j < nint) r.seek(u, j == 0 ? 0 : (uint64_t)bnd[j - 1], j < ctl->nmark ? (int64_t)bnd[j] : (int64_t)ctl->u_len);
    else r.seek(u, 0, -1);
    int pred[3], eobrun;
    const int Al = sc.Al;
    const uint32_t p1 = 1u << Al;
    const int c = sc.comp[0], Ss = sc.Ss, Se = sc.Se;
    const ProgTable &ac = sc.tb[1][0];
    const uint64_t band = bits_range(Ss, Se);
    // the chain over units [u0, u1) of one interval; an MCU that starts after the data ran out is left alone, and so is
    // every later one of the interval
    auto chain = [&](uint64_t u0, uint64_t u1) {
        pred[0] = pred[1] = pred[2] = 0;
        eobrun = 0;
        if (sc.Ss == 0) {
            // ---- DC scans (interleaved: MCU order, every block of the MCU, padding blocks too; or one component)
            UnitWalk wk;
            wk.init(g, sc.comp[0], u0);
            for (uint64_t un = u0; un < u1 && !r.over(); un++, wk.next()) {
                for (int i = 0; i < sc.ncomp; i++) {
                    const int ci = sc.comp[i];
                    const int nb = sc.ncomp > 1 ? (ci ? 1 : g.hs * g.vs) : 1;
                    for (int b = 0; b < nb; b++) {
                        const size_t blk = sc.ncomp > 1 ? (size_t)un * g.bpm + (ci ? g.bpm - 3 + ci : b) : wk.block(g);
                        if (sc.Ah == 0) {          // decode_mcu_DC_first
                            const int s = r.sym(sc.tb[0][i]);
                            const int diff = s ? prog_extend((int)r.get(s), s) : 0;
                            pred[i] += diff;
                            coef[blk * 64] = (int16_t)(pred[i] * (1 << Al));
                        } else if (r.get(1)) {     // decode_mcu_DC_refine: a posted OR on the word that holds coefficient 0
                            atomicOr(reinterpret_cast<unsigned int *>(coef + blk * 64), p1);
                        }
                    }
                }
            }
            return;
        }
        if (sc.Ah == 0) {
            // ---- decode_mcu_AC_first: coefficients by posted stores, new positions OR-ed into the block's mask
            UnitWalk wk;
            wk.init(g, c, u0);
            for (uint64_t un = u0; un < u1 && !r.over(); un++, wk.next()) {
                if (eobrun > 0) { eobrun--; continue; }
                const size_t blk = wk.block(g);
                uint64_t bits = 0;
                for (int k = Ss; k <= Se; k++) {
                    const int rs = r.sym(ac), rr = rs >> 4, ss = rs & 15;
                    if (ss) {
                        k += rr;
                        const int v = prog_extend((int)r.get(ss), ss);
                        if (k <= 63) { coef[blk * 64 + k] = (int16_t)(v * (1 << Al)); bits |= 1ull << k; }
                    } else {
                        if (rr == 15) k += 15;
                        else { eobrun = 1 << rr; if (rr) eobrun += (int)r.get(rr); eobrun--; break; }
                    }
                }
                if (bits) atomicOr(reinterpret_cast<unsigned long long *>(mask + blk), (unsigned long long)bits);
            }
            return;
        }
        // ---- decode_mcu_AC_refine, parsing only: correction bits, new positions and their signs per block
        for (uint64_t un = u0; un < u1; un++) {
            const uint64_t m = cm[un] & band;     // coefficients of the band that are already non-zero
            uint64_t cbits = 0, nm = 0, ns = 0;
            int k = Ss;
            if (r.over()) { corr[un] = 0; newm[un] = 0; news[un] = 0; continue; }
            if (eobrun == 0) {
                while (k <= Se) {
                    const int rs = r.sym(ac), rr = rs >> 4, ss = rs & 15;
                    uint32_t positive = 0;
                    if (ss) positive = r.get(1);                       // the size of a new coefficient is always 1
                    else if (rr != 15) { eobrun = 1 << rr; if (rr) eobrun += (int)r.get(rr); break; }
                    // pass over rr still-zero coefficients, stop at the next one; the non-zero ones on the way take a bit each
                    const uint64_t z = ~m & bits_range(k, Se);
                    const int p = min(select_bit(z, rr), Se + 1);
                    const uint64_t nzs = m & bits_range(k, p - 1);
                    const int n = __popcll(nzs);
                    cbits = (cbits << n) | r.get64(n);
                    if (ss && p <= Se) { nm |= 1ull << p; if (positive) ns |= 1ull << p; }
                    k = p + 1;
                }
            }
            if (eobrun > 0) {
                const int n = __popcll(m & bits_range(k, Se));
                cbits = (cbits << n) | r.get64(n);
                eobrun--;
            }
            corr[un] = cbits; newm[un] = nm; news[un] = ns;
        }
    };
    uint64_t u0 = sc.ri ? (uint64_t)j * sc.ri : 0, u1 = sc.ri ? min(sc.units, u0 + sc.ri) : sc.units;
    for (uint32_t jj = j;; jj++) {
        chain(u0, u1);
        if (jj + 1 != nint || nint >= sc.nint_max) break;
        // interval nint: one MCU of zero bits if this interval ended without running out of data, nothing otherwise
        r.seek(u, ctl->u_len, r.over() ? -1 : (int64_t)ctl->u_len);
        u0 = u1;
        u1 = min(sc.units, u0 + sc.ri);
    }
}

// refinement scans, second half: the parsed words applied to the coefficients, one thread per block
__global__ void __launch_bounds__(256)
k_prog_apply(const uint64_t *__restrict__ cm, const uint64_t *__restrict__ corr, const uint64_t *__restrict__ newm,
             const uint64_t *__restrict__ news, Geom g, int c, uint64_t units, int Ss, int Se, int Al,
             int16_t *__restrict__ coef, uint64_t *__restrict__ mask) {
    const uint64_t u = (uint64_t)blockIdx.x * 256 + threadIdx.x;
    if (u >= units) return;
    const size_t blk = prog_unit_block(g, c, u);
    int16_t *b = coef + blk * 64;
    const int p1 = 1 << Al, m1 = -(1 << Al);
    uint64_t m = cm[u] & bits_range(Ss, Se);
    int i = __popcll(m);
    const uint64_t cb = corr[u];
    while (m) {                                 // ascending positions: the first bit read is the highest of the i bits
        const int k = __ffsll((long long)m) - 1;
        m &= m - 1;
        i--;
        if ((cb >> i) & 1ull) {
            const int v = b[k];
            if ((v & p1) == 0) b[k] = (int16_t)(v + (v >= 0 ? p1 : m1));
        }
    }
    uint64_t nm = newm[u];
    const uint64_t ns = news[u];
    if (nm) mask[blk] |= nm;
    while (nm) {
        const int k = __ffsll((long long)nm) - 1;
        nm &= nm - 1;
        b[k] = (int16_t)(((ns >> k) & 1ull) ? p1 : m1);
    }
}

#define PCK(call)                                                                                                  \
    do {                                                                                                           \
        cudaError_t _e = (call);                                                                                   \
        if (_e != cudaSuccess) {                                                                                   \
            snprintf(err, errlen, "%s at %s:%d", cudaGetErrorString(_e), __FILE__, __LINE__);                       \
            rc = B2J_ECUDA;                                                                                        \
            goto done;                                                                                             \
        }                                                                                                          \
    } while (0)

int dec_progressive(const uint8_t *jpg, size_t len, const JpegInfo &info, const Geom &g, int16_t *d_coef, void *d_tb,
                    uint8_t *d_planes, uint8_t *d_bgr, size_t step, bool gray_out, cudaStream_t s, uint64_t *launches,
                    char *err, size_t errlen, int scale) {
    int rc = B2J_OK;
    uint8_t *d_all = nullptr, *d_file = nullptr, *d_u = nullptr;
    ProgScanDev *d_sc = nullptr;
    ProgCtl *d_ctl = nullptr;
    uint64_t *d_desc = nullptr, *d_mask = nullptr, *d_tmp = nullptr;
    uint32_t *d_bnd = nullptr;
    const int nscans = (int)info.scans.size();
    std::vector<ProgScanDev> hsc(nscans);
    DecTables *htb = nullptr;
    size_t max_seg = 0, max_units = 0, max_int = 1;
    for (int i = 0; i < nscans; i++) {
        const JpegScan &ps = info.scans[i];
        ProgScanDev &sd = hsc[i];
        memset(&sd, 0, sizeof(sd));
        sd.ncomp = ps.ncomp; sd.Ss = ps.Ss; sd.Se = ps.Se; sd.Ah = ps.Ah; sd.Al = ps.Al; sd.ri = ps.restart_interval;
        for (int c = 0; c < ps.ncomp; c++) {
            sd.comp[c] = ps.comp[c];
            const int k = ps.Ss > 0;   // the table the scan decodes with: DC (first DC scans, Ah = 0) or AC
            ProgTable &t = sd.tb[k][c];
            if ((k || ps.Ah == 0) && huff_derive(ps.bits[k][c], ps.vals[k][c], PROG_LUT_BITS, t.lut, t.maxcode, t.valoff, t.vals)) {
                snprintf(err, errlen, "invalid Huffman table in scan %d", i);
                return B2J_EFORMAT;
            }
        }
        sd.units = ps.ncomp > 1 ? (uint64_t)g.mcux * g.mcuy : (uint64_t)g.wib[ps.comp[0]] * g.hib[ps.comp[0]];
        const uint64_t ni = sd.ri ? (sd.units + sd.ri - 1) / sd.ri : 1;
        sd.nint_max = (uint32_t)std::min<uint64_t>(ni, 0x7fffffffu);
        max_seg = std::max(max_seg, ps.seg_len);
        max_units = std::max<size_t>(max_units, (size_t)sd.units);
        max_int = std::max<size_t>(max_int, (size_t)sd.nint_max);
        if (ps.seg_len >= 0xFFFFFFF0ull) { snprintf(err, errlen, "progressive scans of 4 GB and more are not supported"); return B2J_EFORMAT; }
    }
    const size_t ndesc = max_seg / 4096 + 8;
    {   // one allocation for everything the scans need (allocations and frees synchronise: a handful of them per decode
        // would cost more than a small file's kernels)
        auto up = [](size_t x) { return (x + 255) & ~(size_t)255; };
        const size_t o_file = 0, o_u = o_file + up(len + 64), o_sc = o_u + up(max_seg + 4096), o_ctl = o_sc + up(sizeof(ProgScanDev) * nscans),
                     o_desc = o_ctl + up(sizeof(ProgCtl)), o_bnd = o_desc + up(ndesc * 8), o_mask = o_bnd + up((max_int + 2) * 4),
                     o_tmp = o_mask + up((size_t)g.nblocks * 8), total = o_tmp + up(max_units * 8 * 4);
        PCK(cudaMalloc(&d_all, total));
        d_file = d_all + o_file; d_u = d_all + o_u; d_sc = reinterpret_cast<ProgScanDev *>(d_all + o_sc);
        d_ctl = reinterpret_cast<ProgCtl *>(d_all + o_ctl); d_desc = reinterpret_cast<uint64_t *>(d_all + o_desc);
        d_bnd = reinterpret_cast<uint32_t *>(d_all + o_bnd); d_mask = reinterpret_cast<uint64_t *>(d_all + o_mask);
        d_tmp = reinterpret_cast<uint64_t *>(d_all + o_tmp);
    }
    PCK(cudaMemcpyAsync(d_file, jpg, len, cudaMemcpyDefault, s));
    PCK(cudaMemcpyAsync(d_sc, hsc.data(), sizeof(ProgScanDev) * nscans, cudaMemcpyHostToDevice, s));
    PCK(cudaMemsetAsync(d_coef, 0, (size_t)g.nblocks * 128, s));
    PCK(cudaMemsetAsync(d_mask, 0, (size_t)g.nblocks * 8, s));
    for (int i = 0; i < nscans; i++) {
        const JpegScan &ps = info.scans[i];
        const ProgScanDev &sd = hsc[i];
        if (ps.seg_len == 0) continue;
        // front end: stuffing and RSTn markers out, interval starts recorded (the baseline decoder's kernel)
        PCK(cudaMemsetAsync(d_ctl, 0, sizeof(ProgCtl), s));
        PCK(cudaMemsetAsync(d_desc, 0, (ps.seg_len / 4096 + 8) * 8, s));
        PCK(launch_destuff(d_file + ps.seg_off, ps.seg_len, d_u, d_desc, &d_ctl->ticket, 0, destuff_chunks(d_file + ps.seg_off, ps.seg_len), &d_ctl->u_len,
                           &d_ctl->avail, d_bnd, (uint32_t)(max_int + 2), &d_ctl->nmark, &d_ctl->err, s));
        uint64_t *cm = d_tmp, *corr = d_tmp + max_units, *newm = d_tmp + 2 * max_units, *news = d_tmp + 3 * max_units;
        const bool refine_ac = sd.Ss > 0 && sd.Ah > 0;
        const unsigned ugrid = (unsigned)((sd.units + 255) / 256);
        if (refine_ac) {
            k_prog_gather<<<ugrid, 256, 0, s>>>(d_mask, cm, g, sd.comp[0], sd.units);
            PCK(cudaGetLastError());
        }
        k_prog_scan<<<(sd.nint_max + 31) / 32, 32, 0, s>>>(d_u, d_ctl, d_bnd, d_sc + i, g, d_coef, d_mask, cm, corr, newm, news);
        PCK(cudaGetLastError());
        if (refine_ac) {
            k_prog_apply<<<ugrid, 256, 0, s>>>(cm, corr, newm, news, g, sd.comp[0], sd.units, sd.Ss, sd.Se, sd.Al, d_coef, d_mask);
            PCK(cudaGetLastError());
        }
        if (launches) (*launches) += refine_ac ? 4 : 2;
    }
    {   // de-quantisation tables for the back end
        htb = (DecTables *)calloc(1, dec_tables_size());
        if (!htb) { rc = B2J_ENOMEM; goto done; }
        memcpy(htb->q, info.qt, sizeof(htb->q));
        PCK(cudaMemcpyAsync(d_tb, htb, dec_tables_size(), cudaMemcpyHostToDevice, s));
        // the blocks hold their own DCs (dcarr NULL)
        PCK(dec_back_end(d_coef, nullptr, g, d_tb, d_planes, d_bgr, step, gray_out, scale, 0, s, nullptr, nullptr, launches));
    }
    PCK(cudaStreamSynchronize(s));   // the host vectors and the temporary buffers go away below
done:
    if (rc != B2J_OK) cudaStreamSynchronize(s);
    cudaFree(d_all);
    free(htb);
    return rc;
}

}  // namespace b2j
