// scaled_main.cpp -- NvjpegCompressRunner::setDecodeScale: the reference demo's call order (tests/cpp/demo_main.cpp) on
// a CV_8UC3 image with sampling 422 and a CV_8UC1 image with sampling 400, decoded at 1/2, 1/4 and 1/8
// (cv::imread IMREAD_REDUCED_COLOR_d / IMREAD_REDUCED_GRAYSCALE_d); reconstruct() stays full size, an invalid scale gives
// the failure signal and scale 1 the full-size image again.
// usage: scaled W H in.bgr in.gray outdir   -> outdir/{bgr,gray}.jpeg, {bgr,gray}.d{2,4,8}.raw; exit code 0 = every
// run_state, type and size was what it should be
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>

#include "../../include/ImageCompressor.h"

static cv::Mat load(const char *path, int W, int H, int type, int ch) {
    cv::Mat m(H, W, type);
    FILE *f = fopen(path, "rb");
    if (!f || fread(m.data, 1, (size_t)W * H * ch, f) != (size_t)W * H * ch) { fprintf(stderr, "cannot read %s\n", path); exit(2); }
    fclose(f);
    return m;
}

static int run(int W, int H, int sampling, const cv::Mat &image, const std::string &outdir, const std::string &name) {
    const int type = sampling == 400 ? CV_8UC1 : CV_8UC3, ch = sampling == 400 ? 1 : 3;
    int bad = 0, st = 0;
    NvjpegCompressRunner *compressor = new NvjpegCompressRunner(W, H, 95, true, sampling);
    compressor->buildCompressEnv();
    std::vector<unsigned char> obuffer = compressor->compress(image, &st);
    bad += st != 1;
    compressor->deleteCompressEnv();
    compressor->buildDecodeEnv();
    const std::string path = outdir + "/" + name + ".jpeg";
    compressor->save(path, obuffer);
    for (int d : {2, 4, 8}) {
        compressor->setDecodeScale(d);
        cv::Mat r = compressor->decode(path, &st);
        bad += st != 1 || r.type() != type || r.cols != (W + d - 1) / d || r.rows != (H + d - 1) / d;
        FILE *f = fopen((outdir + "/" + name + ".d" + std::to_string(d) + ".raw").c_str(), "wb");
        for (int y = 0; y < r.rows; y++) fwrite(r.data + (size_t)y * r.step, 1, (size_t)r.cols * ch, f);
        fclose(f);
        cv::Mat full = compressor->reconstruct(obuffer, &st);   // full size whatever the decode scale
        bad += st != 1 || full.cols != W || full.rows != H;
    }
    compressor->setDecodeScale(3);
    cv::Mat none = compressor->decode(path, &st);
    bad += st != 0 || !none.empty();
    compressor->setDecodeScale(1);
    cv::Mat full = compressor->decode(path, &st);
    bad += st != 1 || full.cols != W || full.rows != H;
    compressor->deleteDecodeEnv();
    delete compressor;
    return bad;
}

int main(int argc, char *argv[]) {
    if (argc < 6) return 2;
    const int W = atoi(argv[1]), H = atoi(argv[2]);
    const std::string outdir = argv[5];
    int bad = run(W, H, 422, load(argv[3], W, H, CV_8UC3, 3), outdir, "bgr");
    bad += run(W, H, 400, load(argv[4], W, H, CV_8UC1, 1), outdir, "gray");
    return bad ? 1 : EXIT_SUCCESS;
}
