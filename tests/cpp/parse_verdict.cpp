// The product's JPEG header parser (csrc/dec_parse.cpp) on files named on the command line: one line per file,
// "<parse_jpeg rc> <parse_progressive rc> <css>" (css of the parser that accepted the file, -1 if none did).
#include <cstdio>
#include <vector>
#include <cuda_runtime.h>
#include "../../nvjpeg_imagecompressor_b200/csrc/dec.h"
int main(int argc, char **argv) {
    for (int i = 1; i < argc; i++) {
        FILE *f = fopen(argv[i], "rb");
        if (!f) { printf("missing\n"); continue; }
        fseek(f, 0, SEEK_END); long n = ftell(f); rewind(f);
        std::vector<uint8_t> b(n);
        size_t got = fread(b.data(), 1, n, f);
        fclose(f);
        b2j::JpegInfo info;
        b2j::ProgInfo pi;
        const int rb = b2j::parse_jpeg(b.data(), got, &info);
        const int rp = b2j::parse_progressive(b.data(), got, &pi);
        printf("%d %d %d\n", rb, rp, rb == 0 ? info.css : rp == 0 ? pi.css : -1);
        if (rp == 0) b2j::prog_free(&pi);
    }
    return 0;
}
