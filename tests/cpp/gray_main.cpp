// gray_main.cpp -- the reference demo's call order (tests/cpp/demo_main.cpp) with sampling 400 on CV_8UC1 images:
// construct -> buildCompressEnv -> compress x2 (+ a CV_8UC3 image and secondaryCompress, both refused) ->
// deleteCompressEnv -> buildDecodeEnv -> save x2 -> decode x2 -> deleteDecodeEnv -> delete.
// usage: gray W H in1.gray in2.gray outdir     exit code 0 = every run_state was what it should be
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>

#include "../../include/ImageCompressor.h"

static void printState(int run_state) { std::cout << (run_state == 1 ? "[INFO] Successful." : "[INFO] Failed.") << std::endl; }

static cv::Mat load(const char *path, int W, int H) {
    cv::Mat m(H, W, CV_8UC1);
    FILE *f = fopen(path, "rb");
    if (!f || fread(m.data, 1, (size_t)W * H, f) != (size_t)W * H) { fprintf(stderr, "cannot read %s\n", path); exit(2); }
    fclose(f);
    return m;
}

int main(int argc, char *argv[]) {
    if (argc < 6) return 2;
    const int W = atoi(argv[1]), H = atoi(argv[2]);
    const std::string outdir = argv[5];
    int bad = 0, st = 0;
    NvjpegCompressRunner *compressor = new NvjpegCompressRunner(W, H, 95, true, 400);
    int compress_run_state, decode_run_state;
    compressor->buildCompressEnv();
    cv::Mat image1 = load(argv[3], W, H);
    std::vector<unsigned char> obuffer1 = compressor->compress(image1, &compress_run_state);
    printState(compress_run_state); bad += compress_run_state != 1;
    cv::Mat image2 = load(argv[4], W, H);
    std::vector<unsigned char> obuffer2 = compressor->compress(image2, &compress_run_state);
    printState(compress_run_state); bad += compress_run_state != 1;
    cv::Mat bgr(H, W, CV_8UC3);
    memset(bgr.data, 0, bgr.step * H);
    std::vector<unsigned char> wrong = compressor->compress(bgr, &st);   // a BGR image on a gray runner: failure signal
    bad += st != 0 || !wrong.empty();
    std::vector<unsigned char> diffjpg; cv::Mat rec; double ps = 0;
    std::vector<unsigned char> sec = compressor->secondaryCompress(image1, &diffjpg, &rec, &ps, true, &st);
    bad += st != 0 || !sec.empty();
    compressor->deleteCompressEnv();

    compressor->buildDecodeEnv();
    const std::string p1 = outdir + "/1.jpeg", p2 = outdir + "/2.jpeg";
    compressor->save(p1, obuffer1);
    compressor->save(p2, obuffer2);
    cv::Mat d1 = compressor->decode(p1, &decode_run_state);
    printState(decode_run_state); bad += decode_run_state != 1 || d1.type() != CV_8UC1;
    cv::Mat d2 = compressor->reconstruct(obuffer2, &decode_run_state);
    printState(decode_run_state); bad += decode_run_state != 1 || d2.type() != CV_8UC1;
    FILE *f = fopen((outdir + "/1.dec.gray").c_str(), "wb"); fwrite(d1.data, 1, d1.total(), f); fclose(f);
    f = fopen((outdir + "/2.dec.gray").c_str(), "wb"); fwrite(d2.data, 1, d2.total(), f); fclose(f);
    compressor->deleteDecodeEnv();
    delete compressor;

    NvjpegCompressRunner *multi = new NvjpegCompressRunner(W, H, 95, true, 400, 2);   // gray over two GPUs: refused
    multi->buildCompressEnv();
    std::vector<unsigned char> none = multi->compress(image1, &st);
    bad += st != 0 || !none.empty();
    delete multi;
    return bad ? 1 : EXIT_SUCCESS;
}
