// ImageCompressor.h -- drop-in C++ facade with the reference's public interface
// (OroChippw/Nvjpeg-ImageCompressor src/ImageCompressorDll/ImageCompressor.h:22-42): same class name, constructor
// defaults, method names, argument meaning and failure convention (empty result + *run_state = 0). The body
// (facade/ImageCompressor.cpp) forwards to the extern "C" engine in libb2jpeg.so instead of nvJPEG.
//
// Differences a maintainer should know (all additive):
//   * the sampling factor the reference hard-codes (ImageCompressorImpl.cu:31) is a defaulted 5th constructor argument
//     (README default 4:2:2) and the stream is baseline sequential, not progressive (ImageCompressorImpl.cu:28)
//   * CUDA failures never exit(1) (ImageCompressorImpl.cuh:16-34); they produce the documented failure signal
//   * reconstruct / differenceMap / psnr / secondaryCompress implement the README's feature bullet (README.md:8)
//   * a defaulted 6th constructor argument spreads compress() over several GPUs; setRestartRows() turns DRI/RSTn on;
//     setDecodeScale() makes decode() return a reduced image (cv::IMREAD_REDUCED_*)
#ifndef IMAGECOMPRESSOR_H_
#define IMAGECOMPRESSOR_H_

#include <iostream>
#include <string>
#include <vector>

#if defined(B2J_USE_CV_SHIM) || !__has_include(<opencv2/core.hpp>)
#include "cv_shim.h"
#else
#include <opencv2/core.hpp>
#endif

#if defined(_WIN32)
#ifdef NVJPEG_COMPRESS_RUNNER_EXPORTS
#define NVJPEG_COMPRESS_RUNNER_API __declspec(dllexport)
#else
#define NVJPEG_COMPRESS_RUNNER_API __declspec(dllimport)
#endif
#else
#define NVJPEG_COMPRESS_RUNNER_API __attribute__((visibility("default")))
#endif

class NvjpegCompressRunnerImpl;

class NVJPEG_COMPRESS_RUNNER_API NvjpegCompressRunner {
private:
    NvjpegCompressRunnerImpl *compressor;

public:
    // sampling: 444, 422, 440, 420, 411, or 400 (gray: compress() takes CV_8UC1, decode() / reconstruct() return CV_8UC1
    // -- the one-component file, or the Y plane of a colour file; secondaryCompress() and ngpus > 1 are not available
    // and give the failure signal). ngpus > 1: compress() cuts the image into MCU-row strips over that many GPUs of
    // this node (devices 0 .. ngpus-1, or the comma-separated list in B2J_MULTI_DEVICES) from this one process
    // (b2j_multi_*); the bytes are the single-GPU bytes.
    NvjpegCompressRunner(int width = 8320, int height = 40000, int quality = 95, bool optimize = true, int sampling = 422,
                         int ngpus = 1);
    ~NvjpegCompressRunner();

    NvjpegCompressRunner(const NvjpegCompressRunner &) = delete;
    NvjpegCompressRunner &operator=(const NvjpegCompressRunner &) = delete;

    // CV_8UC3 BGR pixels (CV_8UC1 with sampling 400; any row step) -> complete JFIF bytes. Empty vector and
    // *run_state = 0 on failure (empty, oversized or wrongly typed image, CUDA error), 1 on success; run_state may be null. Replaces ImageCompressor.cpp:45-61 /
    // ImageCompressorImpl.cu:269-294 (cv::split + 3 x cudaMemcpy + nvjpegEncodeImage + retrieve): b2j_encode, pageable
    // pixels are staged by the engine's copy threads. Prints the reference's "[INFO] ... Cost Time" line unless B2J_QUIET=1.
    std::vector<unsigned char> compress(cv::Mat image, int *run_state);
    // JPEG file -> CV_8UC3 BGR. Empty Mat and *run_state = 0 when the file cannot be opened or decoded
    // (ImageCompressor.cpp:63-88, ImageCompressorImpl.cu:311-385 + getCVImageOnCPU :184-232): b2j_decode, the
    // planar->interleaved step happens in the kernel's store.
    cv::Mat decode(std::string image_path, int *run_state);
    // Binary write of the bytes (ImageCompressor.cpp:90-101; the size is not narrowed to int here).
    void save(std::string save_path, std::vector<unsigned char> obuffer);

    // The reference's environment protocol (ImageCompressor.h:38-41): build before use, delete when done. Here one
    // engine context serves both directions; building twice is harmless, using an unbuilt environment fails cleanly
    // (*run_state = 0) instead of dereferencing uninitialised nvJPEG handles.
    void buildCompressEnv();
    void buildDecodeEnv();
    void deleteCompressEnv();
    void deleteDecodeEnv();

    // Restart markers every `mcu_rows` MCU rows in what compress() writes (0 = none, the default; single-GPU path):
    // nvjpegEncoderParamsSetRestartInterval / cv2 IMWRITE_JPEG_RST_INTERVAL at the reference's parameter site
    // (ImageCompressorImpl.cu:28-31). decode() / reconstruct() accept any restart interval and progressive files.
    void setRestartRows(int mcu_rows);
    // decode() returns the image at 1 / denom (denom 1, 2, 4 or 8; 1 = full size, the default), as
    // cv::imread(path, IMREAD_REDUCED_COLOR_denom) does (IMREAD_REDUCED_GRAYSCALE_denom with sampling 400): libjpeg's DCT
    // scaling, ceil(W / denom) x ceil(H / denom) pixels. Any other value makes decode() give the failure signal.
    // reconstruct() stays full size (differenceMap / psnr compare it with the original).
    void setDecodeScale(int denom);

    // README.md:8 -- reconstruction, difference map, secondary compression, PSNR
    cv::Mat reconstruct(const std::vector<unsigned char> &obuffer, int *run_state);
    cv::Mat differenceMap(cv::Mat a, cv::Mat b, bool offset128, int *run_state);
    double psnr(cv::Mat a, cv::Mat b, int *run_state);
    // returns the JPEG of `image`; diff_jpeg receives the JPEG of the difference map (orig vs reconstruction)
    std::vector<unsigned char> secondaryCompress(cv::Mat image, std::vector<unsigned char> *diff_jpeg, cv::Mat *reconstruction,
                                                 double *psnr_db, bool offset128, int *run_state);
};

#endif  // IMAGECOMPRESSOR_H_
