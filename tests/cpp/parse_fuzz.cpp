// ASAN fuzz harness for the product's JPEG header parser (csrc/dec_parse.cpp: parse_jpeg, dec_build_tables, huff_derive):
// every mutated input is copied into an exact-size heap block so that any read past the end is reported.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>
#include <cuda_runtime.h>
#include "../../nvjpeg_imagecompressor_b200/csrc/dec.h"
#include "../../nvjpeg_imagecompressor_b200/csrc/dec_kernels.h"
static uint32_t st = 99;
static uint32_t rnd() { st = st * 1664525u + 1013904223u; return st >> 8; }
int main(int argc, char **argv) {
    const int iters = argc > 1 ? atoi(argv[1]) : 100000;
    std::vector<std::vector<uint8_t>> seeds;
    for (int i = 2; i < argc; i++) {
        FILE *f = fopen(argv[i], "rb"); if (!f) continue;
        fseek(f, 0, SEEK_END); long n = ftell(f); rewind(f);
        std::vector<uint8_t> b(n); if (fread(b.data(), 1, n, f) != (size_t)n) { fclose(f); continue; } fclose(f);
        seeds.push_back(b);
    }
    long ok = 0, total = 0;
    for (int it = 0; it < iters; it++) {
        std::vector<uint8_t> s = seeds[it % seeds.size()];
        size_t hdr = s.size() < 900 ? s.size() : 900;
        switch (it % 5) {
        case 0: s.resize(rnd() % (s.size() + 1)); break;
        case 1: for (int k = 0, n = 1 + rnd() % 6; k < n; k++) s[rnd() % hdr] = (uint8_t)rnd(); break;
        case 2: { size_t i = rnd() % hdr; s.insert(s.begin() + i, 1 + rnd() % 40, (uint8_t)rnd()); break; }
        case 3: { size_t i = 2 + rnd() % (hdr - 6); s[i] = 0xFF; s[i + 1] = 0xC0 + rnd() % 0x3F; s[i + 2] = (uint8_t)rnd(); s[i + 3] = (uint8_t)rnd(); break; }
        case 4: { size_t i = 2 + rnd() % (hdr - 6); s[i + 2] = 0xFF; s[i + 3] = 0xFF; break; }   // huge segment lengths
        }
        uint8_t *heap = (uint8_t *)malloc(s.size() ? s.size() : 1);
        memcpy(heap, s.data(), s.size());
        b2j::JpegInfo info;
        int rc = b2j::parse_jpeg(heap, s.size(), &info);
        if (rc == 0) {
            ok++;
            if (info.W <= 0 || info.H <= 0 || info.css < 0 || info.css > 4 || info.scans.empty()) { printf("BAD INFO it=%d\n", it); return 2; }
            for (const b2j::JpegScan &sc : info.scans)
                if (sc.seg_off + sc.seg_len > s.size() || sc.ncomp < 1 || sc.ncomp > 3) { printf("BAD SCAN it=%d\n", it); return 2; }
            // the table builders write fixed-size blocks: exact-size heap copies so ASAN sees any overflow
            if (!info.progressive) {
                void *tb = malloc(b2j::dec_tables_size());
                b2j::dec_build_tables(info, tb);
                free(tb);
            } else {   // dec_prog.cu: one table per component and class of every scan
                for (const b2j::JpegScan &sc : info.scans)
                    for (int k = 0; k < 2; k++)
                        for (int c = 0; c < sc.ncomp; c++) {
                            uint16_t *lut = (uint16_t *)malloc(sizeof(uint16_t) << b2j::PROG_LUT_BITS);
                            int32_t *maxcode = (int32_t *)malloc(18 * 4), *valoff = (int32_t *)malloc(17 * 4);
                            uint8_t *vals = (uint8_t *)malloc(256);
                            b2j::huff_derive(sc.bits[k][c], sc.vals[k][c], b2j::PROG_LUT_BITS, lut, maxcode, valoff, vals);
                            free(lut); free(maxcode); free(valoff); free(vals);
                        }
            }
        }
        total++;
        free(heap);
    }
    printf("inputs %ld accepted %ld\n", total, ok);
    return 0;
}
