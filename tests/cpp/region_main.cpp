// region_main.cpp -- NvjpegCompressRunner::setDecodeRegion: the reference demo's call order (tests/cpp/demo_main.cpp) on
// a CV_8UC3 image with sampling 422 and a CV_8UC1 image with sampling 400, decoded as one rectangle at scales 1 and 4;
// reconstruct() stays full size, an invalid region and one outside the image give the failure signal, and (0, 0, 0, 0)
// the whole image again.
// usage: region W H in.bgr in.gray outdir   -> outdir/{bgr,gray}.jpeg, {bgr,gray}.s{1,4}.raw (the rectangles of
// REGIONS); exit code 0 = every run_state, type and size was what it should be
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>

#include "../../include/ImageCompressor.h"

// scale, x, y, w, h (tests/test_gpu_facade_region.py crops the CPU checker's output with the same numbers)
static const int REGIONS[2][5] = {{1, 37, 21, 200, 100}, {4, 3, 5, 50, 40}};

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
    for (const auto &r : REGIONS) {
        compressor->setDecodeScale(r[0]);
        compressor->setDecodeRegion(r[1], r[2], r[3], r[4]);
        cv::Mat m = compressor->decode(path, &st);
        bad += st != 1 || m.type() != type || m.cols != r[3] || m.rows != r[4];
        FILE *f = fopen((outdir + "/" + name + ".s" + std::to_string(r[0]) + ".raw").c_str(), "wb");
        for (int y = 0; y < m.rows; y++) fwrite(m.data + (size_t)y * m.step, 1, (size_t)m.cols * ch, f);
        fclose(f);
        cv::Mat full = compressor->reconstruct(obuffer, &st);   // full size whatever the decode region
        bad += st != 1 || full.cols != W || full.rows != H;
    }
    compressor->setDecodeScale(1);
    compressor->setDecodeRegion(-1, 0, 8, 8);   // invalid
    cv::Mat none = compressor->decode(path, &st);
    bad += st != 0 || !none.empty();
    compressor->setDecodeRegion(W - 7, 0, 8, 8);   // one column outside the image
    none = compressor->decode(path, &st);
    bad += st != 0 || !none.empty();
    compressor->setDecodeRegion(0, 0, 0, 0);
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
