// facade/ImageCompressor.cpp -- NvjpegCompressRunner over the C-ABI (include/b2jpeg.h). Compile this file into the
// host application (or its own shared library) against the application's OpenCV; it needs only libb2jpeg.so.
// Mirrors the reference's ImageCompressor.cpp:14-101 (timing print, run_state convention, save()).
#include "../include/ImageCompressor.h"

#include <chrono>
#include <cstdio>
#include <fstream>

#include "../include/b2jpeg.h"

class NvjpegCompressRunnerImpl {
public:
    b2j_params p;
    b2j_ctx *enc = nullptr, *dec = nullptr;
    int ngpus = 1, restart_rows = 0;
    int decode_scale = 1;         // setDecodeScale: decode() returns the image at 1 / decode_scale
    b2j_multi *multi = nullptr;   // compress() over several GPUs (ngpus > 1)
    static bool quiet() { return getenv("B2J_QUIET") != nullptr; }
    int ensure(b2j_ctx **c) {
        if (*c) return 0;
        if (enc) { *c = enc; return 0; }
        if (dec) { *c = dec; return 0; }
        return b2j_create(&p, c);
    }
    void drop(b2j_ctx **c, b2j_ctx *other) {
        if (*c && *c != other) b2j_destroy(*c);
        *c = nullptr;
    }
    b2j_ctx *any() { return enc ? enc : dec; }
    bool gray() const { return p.css == B2J_CSS_GRAY; }
    int mat_type() const { return gray() ? CV_8UC1 : CV_8UC3; }   // what compress() takes and decode() returns
};

static int css_of(int sampling) {
    switch (sampling) {
    case 444: return B2J_CSS_444;
    case 440: return B2J_CSS_440;
    case 420: return B2J_CSS_420;
    case 411: return B2J_CSS_411;
    case 400: return B2J_CSS_GRAY;
    default: return B2J_CSS_422;
    }
}

NvjpegCompressRunner::NvjpegCompressRunner(int width, int height, int quality, bool optimize, int sampling, int ngpus) {
    compressor = new NvjpegCompressRunnerImpl();
    compressor->ngpus = ngpus < 1 ? 1 : ngpus;
    b2j_default_params(&compressor->p);
    compressor->p.width = width; compressor->p.height = height; compressor->p.quality = quality;
    compressor->p.optimize = optimize ? 1 : 0; compressor->p.css = css_of(sampling);
}

NvjpegCompressRunner::~NvjpegCompressRunner() {
    deleteCompressEnv();
    deleteDecodeEnv();
    delete compressor;
    if (!NvjpegCompressRunnerImpl::quiet()) std::cout << "[INFO] Delete NvjpegCompressRunnerImpl Successfully ..." << std::endl;
}

void NvjpegCompressRunner::buildCompressEnv() {
    if (compressor->ensure(&compressor->enc) != 0) std::cerr << "[ERROR] buildCompressEnv: no CUDA device / out of memory" << std::endl;
    else b2j_set_restart_rows(compressor->enc, compressor->restart_rows);
    if (compressor->ngpus > 1 && compressor->gray()) {   // the strips assume three components: compress() fails instead
        std::cerr << "[ERROR] buildCompressEnv: gray (400) images are not encoded over several GPUs" << std::endl;
        compressor->drop(&compressor->enc, compressor->dec);
        return;
    }
    if (compressor->ngpus > 1 && !compressor->multi) {
        int ids[16], n = 0;
        if (const char *e = getenv("B2J_MULTI_DEVICES")) {   // e.g. "0,1,2,3" (tests: "0,0" = two contexts on one GPU)
            for (const char *q = e; *q && n < 16;) { ids[n++] = atoi(q); while (*q && *q != ',') q++; if (*q == ',') q++; }
        } else {
            for (; n < compressor->ngpus && n < 16; n++) ids[n] = n;
        }
        if (b2j_multi_create(&compressor->p, n, ids, &compressor->multi) != 0) {
            std::cerr << "[ERROR] buildCompressEnv: cannot set up " << n << " GPUs, using one" << std::endl;
            compressor->multi = nullptr;
        }
    }
}
void NvjpegCompressRunner::setRestartRows(int mcu_rows) {
    compressor->restart_rows = mcu_rows < 0 ? 0 : mcu_rows;
    if (compressor->enc) b2j_set_restart_rows(compressor->enc, compressor->restart_rows);
}
void NvjpegCompressRunner::buildDecodeEnv() {
    if (compressor->ensure(&compressor->dec) != 0) std::cerr << "[ERROR] buildDecodeEnv: no CUDA device / out of memory" << std::endl;
}
void NvjpegCompressRunner::deleteCompressEnv() {
    if (compressor->multi) { b2j_multi_destroy(compressor->multi); compressor->multi = nullptr; }
    compressor->drop(&compressor->enc, compressor->dec);
}
void NvjpegCompressRunner::deleteDecodeEnv() { compressor->drop(&compressor->dec, compressor->enc); }

std::vector<unsigned char> NvjpegCompressRunner::compress(cv::Mat image, int *run_state) {
    auto t0 = std::chrono::steady_clock::now();
    std::vector<unsigned char> obuffer;
    b2j_ctx *c = compressor->enc;
    if (c && !image.empty() && image.type() == compressor->mat_type()) {
        size_t n = 0;
        int rc;
        if (compressor->multi && compressor->restart_rows == 0) {
            // strips over several GPUs: encode, size the vector to the stitched stream, fetch every strip's bytes into place
            rc = b2j_multi_encode_begin(compressor->multi, image.data, image.step, image.cols, image.rows, &n);
            if (rc == B2J_OK) { obuffer.resize(n); rc = b2j_multi_encode_fetch(compressor->multi, obuffer.data(), n); }
            if (rc != B2J_OK) { std::cerr << "[ERROR] compress: " << b2j_multi_last_error(compressor->multi) << std::endl; n = 0; }
        } else {
            // encode first, then size the vector to the JPEG (no zero-filled worst-case buffer), then fetch the bytes
            rc = b2j_encode_begin(c, image.data, image.step, image.cols, image.rows, &n);
            if (rc == B2J_OK) { obuffer.resize(n); rc = b2j_encode_fetch(c, obuffer.data(), n); }
            if (rc != B2J_OK) { std::cerr << "[ERROR] compress: " << b2j_last_error(c) << std::endl; n = 0; }
        }
        obuffer.resize(n);
    }
    if (run_state) *run_state = obuffer.empty() ? 0 : 1;
    auto ms = std::chrono::duration_cast<std::chrono::milliseconds>(std::chrono::steady_clock::now() - t0).count();
    if (!NvjpegCompressRunnerImpl::quiet()) std::cout << "[INFO] NvjpegCompressRunner Compress Func Cost Time : " << ms << " ms" << std::endl;
    return obuffer;
}

// JPEG bytes -> pixels at 1 / scale. The scale is set on the (possibly shared) context for this call only: compress()
// and reconstruct() keep seeing full-size decodes.
static cv::Mat decode_at(NvjpegCompressRunnerImpl *m, const std::vector<unsigned char> &jpg, int scale) {
    cv::Mat result;
    b2j_ctx *c = m->dec ? m->dec : m->enc;
    if (!c || jpg.empty()) return result;
    if (b2j_set_decode_scale(c, scale) != B2J_OK) {
        std::cerr << "[ERROR] decode: invalid decode scale " << scale << " (1, 2, 4 or 8)" << std::endl;
        return result;
    }
    int w = 0, h = 0;
    if (b2j_decode(c, jpg.data(), jpg.size(), nullptr, 0, &w, &h) == B2J_OK) {
        result.create(h, w, m->mat_type());
        if (b2j_decode(c, jpg.data(), jpg.size(), result.data, result.step, &w, &h) != B2J_OK) {
            std::cerr << "[ERROR] decode: " << b2j_last_error(c) << std::endl;
            result = cv::Mat();
        }
    }
    b2j_set_decode_scale(c, 1);
    return result;
}

cv::Mat NvjpegCompressRunner::reconstruct(const std::vector<unsigned char> &jpg, int *run_state) {
    cv::Mat result = decode_at(compressor, jpg, 1);   // full size: differenceMap / psnr compare it with the original
    if (run_state) *run_state = result.empty() ? 0 : 1;
    return result;
}

void NvjpegCompressRunner::setDecodeScale(int denom) { compressor->decode_scale = denom; }

cv::Mat NvjpegCompressRunner::decode(std::string image_path, int *run_state) {
    FILE *f = fopen(image_path.c_str(), "rb");
    if (!f) {
        std::cerr << "Failed to open JPEG file." << std::endl;
        if (run_state) *run_state = 0;
        return cv::Mat();
    }
    auto t0 = std::chrono::steady_clock::now();
    fseek(f, 0, SEEK_END);
    const long sz = ftell(f);
    rewind(f);
    std::vector<unsigned char> jpg(sz > 0 ? (size_t)sz : 0);
    const size_t rd = jpg.empty() ? 0 : fread(jpg.data(), 1, jpg.size(), f);
    fclose(f);
    cv::Mat result;
    if (rd == jpg.size() && !jpg.empty()) result = decode_at(compressor, jpg, compressor->decode_scale);
    else std::cerr << "[INFO] Failed to read the entire JPEG data." << std::endl;
    if (run_state) *run_state = result.empty() ? 0 : 1;
    auto ms = std::chrono::duration_cast<std::chrono::milliseconds>(std::chrono::steady_clock::now() - t0).count();
    if (!NvjpegCompressRunnerImpl::quiet()) std::cout << "[INFO] NvjpegCompressRunner Decode Func Cost Time : " << ms << " ms" << std::endl;
    return result;
}

void NvjpegCompressRunner::save(std::string save_path, std::vector<unsigned char> obuffer) {
    try {
        std::ofstream out(save_path, std::ios::out | std::ios::binary);
        out.write(reinterpret_cast<const char *>(obuffer.data()), (std::streamsize)obuffer.size());
        out.close();
    } catch (const std::exception &e) {
        std::cerr << "Exception caught: " << e.what() << std::endl;
    }
}

static bool same_shape(const cv::Mat &a, const cv::Mat &b) {
    return !a.empty() && !b.empty() && a.rows == b.rows && a.cols == b.cols && a.type() == b.type() && a.isContinuous() && b.isContinuous();
}

cv::Mat NvjpegCompressRunner::differenceMap(cv::Mat a, cv::Mat b, bool offset128, int *run_state) {
    cv::Mat out;
    b2j_ctx *c = compressor->any();
    if (c && same_shape(a, b)) {
        out.create(a.rows, a.cols, a.type());
        if (b2j_diff(c, a.data, b.data, a.total() * a.elemSize(), offset128 ? B2J_DIFF_OFFSET128 : B2J_DIFF_ABS, out.data) != B2J_OK) out = cv::Mat();
    }
    if (run_state) *run_state = out.empty() ? 0 : 1;
    return out;
}

double NvjpegCompressRunner::psnr(cv::Mat a, cv::Mat b, int *run_state) {
    double v = 0;
    b2j_ctx *c = compressor->any();
    const bool ok = c && same_shape(a, b) && b2j_psnr(c, a.data, b.data, a.total() * a.elemSize(), &v, nullptr) == B2J_OK;
    if (run_state) *run_state = ok ? 1 : 0;
    return ok ? v : 0.0;
}

std::vector<unsigned char> NvjpegCompressRunner::secondaryCompress(cv::Mat image, std::vector<unsigned char> *diff_jpeg, cv::Mat *reconstruction,
                                                                   double *psnr_db, bool offset128, int *run_state) {
    std::vector<unsigned char> j1, j2;
    b2j_ctx *c = compressor->gray() ? nullptr : compressor->enc;   // not on gray contexts (b2j_secondary refuses them)
    if (c && !image.empty() && image.type() == CV_8UC3) {
        // device resident: upload once, both encodes and the reconstruction stay in HBM; the host vectors are sized to
        // the two streams after the fact (b2j_secondary_device / _finish), the pixels come down only if asked for
        std::vector<unsigned char> none;
        size_t n1 = 0, n2 = 0;
        double ps = 0;
        const size_t row = (size_t)image.cols * 3;
        int rc = b2j_secondary(c, image.data, image.step, image.cols, image.rows, offset128 ? B2J_DIFF_OFFSET128 : B2J_DIFF_ABS, nullptr, 0, &n1,
                               nullptr, 0, &n2, nullptr, 0, &ps);
        if (rc == B2J_OK) {
            j1.resize(n1);
            j2.resize(n2);
            cv::Mat rec;
            if (reconstruction) rec.create(image.rows, image.cols, CV_8UC3);
            rc = b2j_secondary_fetch(c, j1.data(), n1, j2.data(), n2, reconstruction ? rec.data : nullptr, reconstruction ? (size_t)rec.step : row);
            if (rc == B2J_OK && reconstruction) *reconstruction = rec;
        }
        if (rc != B2J_OK) { std::cerr << "[ERROR] secondaryCompress: " << b2j_last_error(c) << std::endl; j1.clear(); j2.clear(); }
        if (diff_jpeg) *diff_jpeg = j2;
        if (psnr_db) *psnr_db = ps;
    }
    if (run_state) *run_state = j1.empty() ? 0 : 1;
    return j1;
}
