// The product's JPEG header parser (csrc/dec_parse.cpp) on files named on the command line: one line per file,
// "<parse_jpeg rc> <progressive> <css>" (progressive and css as parsed, 0 and -1 for a refused file).
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
        const int rc = b2j::parse_jpeg(b.data(), got, &info);
        printf("%d %d %d\n", rc, rc == 0 && info.progressive ? 1 : 0, rc == 0 ? info.css : -1);
    }
    return 0;
}
