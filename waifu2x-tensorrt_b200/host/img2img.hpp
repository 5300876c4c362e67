// Header-only C++ shim that re-creates the reference's operator surface on top of the C ABI (include/w2x.h):
//   namespace trt { enum class Precision; struct BuildConfig; struct RenderConfig; enum Severity;
//                   using MessageCallback / ProgressCallback; class Img2Img { build, load, render, set*Callback }; }
// Field names, defaults, argument meaning and the bool error convention follow
// /root/reference/src/tensorrt/{config.h:7-43, logger.h:11-21, img2img.h:14-50}.  OpenCV is not required: `render`
// takes raw BGR8 pointers + strides; when <opencv2/core.hpp> has been included first, the cv::Mat overload with the
// reference's exact signature (img2img.h:20) is available too.
#pragma once
#include <functional>
#include <string>
#include <utility>
#include <vector>

#include "../../include/w2x.h"

namespace trt {

enum class Precision { TF32, FP16 };  // config.h:7-10

struct Point2d {  // stands in for cv::Point2d (config.h:41)
    double x = 0, y = 0;
    Point2d() = default;
    Point2d(double x_, double y_) : x(x_), y(y_) {}
};

struct BuildConfig {  // config.h:12-31
    int deviceId = 0;
    Precision precision = Precision::FP16;
    int minBatchSize = 1, optBatchSize = 1, maxBatchSize = 4;
    int minChannels = 3, optChannels = 3, maxChannels = 3;
    int minWidth = 64, optWidth = 256, maxWidth = 640;
    int minHeight = 64, optHeight = 256, maxHeight = 640;
};

struct RenderConfig {  // config.h:33-43
    int deviceId = 0;
    Precision precision = Precision::FP16;
    int batchSize = 1;
    int channels = 3;
    int height = 256;
    int width = 256;
    int scaling = 4;
    Point2d overlap = Point2d(0.0625, 0.0625);
    bool tta = false;
};

enum Severity { critical, error, warn, info, debug, trace };  // logger.h:11-18

using MessageCallback = std::function<void(Severity, const std::string&)>;  // logger.h:20
using ProgressCallback = std::function<void(int, int, double)>;             // logger.h:21

class Img2Img {
public:
    Img2Img() : h_(w2x_create()) {}
    virtual ~Img2Img() { w2x_destroy(h_); }
    Img2Img(const Img2Img&) = delete;
    Img2Img& operator=(const Img2Img&) = delete;

    bool build(const std::string& path, const BuildConfig& c) {
        w2x_build_config b{c.deviceId, c.precision == Precision::FP16 ? W2X_PRECISION_FP16 : W2X_PRECISION_TF32,
                           c.minBatchSize, c.optBatchSize, c.maxBatchSize, c.minChannels, c.optChannels, c.maxChannels,
                           c.minWidth, c.optWidth, c.maxWidth, c.minHeight, c.optHeight, c.maxHeight};
        return w2x_build(h_, path.c_str(), &b) != 0;
    }

    bool load(const std::string& path, const RenderConfig& c) {
        w2x_render_config r{c.deviceId, c.precision == Precision::FP16 ? W2X_PRECISION_FP16 : W2X_PRECISION_TF32,
                            c.batchSize, c.channels, c.height, c.width, c.scaling, c.overlap.x, c.overlap.y, c.tta ? 1 : 0};
        scaling_ = c.scaling;
        return w2x_load(h_, path.c_str(), &r) != 0;
    }

    // BGR8 HWC in, BGR8 HWC out ((width*scaling) x (height*scaling)); caller owns both buffers (main.cpp:228-235)
    bool render(const unsigned char* srcBgr, int width, int height, size_t srcStride, unsigned char* dstBgr, size_t dstStride) {
        return w2x_render(h_, srcBgr, width, height, srcStride, dstBgr, dstStride) != 0;
    }

#ifdef OPENCV_CORE_HPP
    // the reference signature (img2img.h:20); dst is (re)created like GpuMat::download would
    bool render(const cv::Mat& src, cv::Mat& dst) {
        if (src.type() != CV_8UC3) return false;
        dst.create(src.rows * scaling_, src.cols * scaling_, CV_8UC3);
        return render(src.data, src.cols, src.rows, src.step, dst.data, dst.step);
    }
#endif

    void setMessageCallback(MessageCallback cb) {
        msg_ = std::move(cb);
        w2x_set_message_callback(h_, msg_ ? &Img2Img::onMessage : nullptr, this);
    }
    void setProgressCallback(ProgressCallback cb) {
        prog_ = std::move(cb);
        w2x_set_progress_callback(h_, prog_ ? &Img2Img::onProgress : nullptr, this);
    }

    // extensions (not in the reference): BGRA8 HWC in, BGRA8 HWC out, synchronous, see w2x_render_bgra in include/w2x.h
    bool renderBgra(const unsigned char* srcBgra, int width, int height, size_t srcStride, unsigned char* dstBgra, size_t dstStride) {
        return w2x_render_bgra(h_, srcBgra, width, height, srcStride, dstBgra, dstStride) != 0;
    }

    // up to three frames in flight, see w2x_submit / w2x_wait in include/w2x.h
    int submit(const unsigned char* srcBgr, int width, int height, size_t srcStride, unsigned char* dstBgr, size_t dstStride) {
        return w2x_submit(h_, srcBgr, width, height, srcStride, dstBgr, dstStride);
    }

    // extensions: the output reduced to dstWidth x dstHeight (at most the model's scale), see w2x_render_resized in include/w2x.h
    bool renderResized(const unsigned char* srcBgr, int width, int height, size_t srcStride, unsigned char* dstBgr, int dstWidth, int dstHeight,
                       size_t dstStride) {
        return w2x_render_resized(h_, srcBgr, width, height, srcStride, dstBgr, dstWidth, dstHeight, dstStride) != 0;
    }
    int submitResized(const unsigned char* srcBgr, int width, int height, size_t srcStride, unsigned char* dstBgr, int dstWidth, int dstHeight,
                      size_t dstStride) {
        return w2x_submit_resized(h_, srcBgr, width, height, srcStride, dstBgr, dstWidth, dstHeight, dstStride);
    }
    // extensions: 16 bits per channel, native-endian u16 BGR in and out, strides in bytes, see w2x_render_u16 in include/w2x.h
    bool renderU16(const uint16_t* srcBgr, int width, int height, size_t srcStride, uint16_t* dstBgr, size_t dstStride) {
        return w2x_render_u16(h_, srcBgr, width, height, srcStride, dstBgr, dstStride) != 0;
    }
    int submitU16(const uint16_t* srcBgr, int width, int height, size_t srcStride, uint16_t* dstBgr, size_t dstStride) {
        return w2x_submit_u16(h_, srcBgr, width, height, srcStride, dstBgr, dstStride);
    }
    bool wait(int ticket) { return w2x_wait(h_, ticket) != 0; }

    w2x_engine* handle() const { return h_; }

private:
    static void onMessage(int sev, const char* m, void* self) { static_cast<Img2Img*>(self)->msg_(static_cast<Severity>(sev), m); }
    static void onProgress(int cur, int tot, double speed, void* self) { static_cast<Img2Img*>(self)->prog_(cur, tot, speed); }
    w2x_engine* h_;
    int scaling_ = 1;
    MessageCallback msg_;
    ProgressCallback prog_;
};

// Frame-parallel multi-GPU extension (w2x_pool_*, include/w2x.h): same build / load / submit / wait shape as Img2Img, one engine per
// listed device, frame f -> devices[f % n].  The message callback may fire on the pool's worker threads.
class Img2ImgPool {
public:
    explicit Img2ImgPool(const std::vector<int>& devices) : h_(w2x_pool_create(devices.data(), (int)devices.size())) {}
    ~Img2ImgPool() { w2x_pool_destroy(h_); }
    Img2ImgPool(const Img2ImgPool&) = delete;
    Img2ImgPool& operator=(const Img2ImgPool&) = delete;
    bool valid() const { return h_ != nullptr; }
    bool build(const std::string& path, const BuildConfig& c) {
        w2x_build_config b{c.deviceId, c.precision == Precision::FP16 ? W2X_PRECISION_FP16 : W2X_PRECISION_TF32,
                           c.minBatchSize, c.optBatchSize, c.maxBatchSize, c.minChannels, c.optChannels, c.maxChannels,
                           c.minWidth, c.optWidth, c.maxWidth, c.minHeight, c.optHeight, c.maxHeight};
        return w2x_pool_build(h_, path.c_str(), &b) != 0;
    }
    bool load(const std::string& path, const RenderConfig& c) {
        w2x_render_config r{c.deviceId, c.precision == Precision::FP16 ? W2X_PRECISION_FP16 : W2X_PRECISION_TF32,
                            c.batchSize, c.channels, c.height, c.width, c.scaling, c.overlap.x, c.overlap.y, c.tta ? 1 : 0};
        return w2x_pool_load(h_, path.c_str(), &r) != 0;
    }
    int submit(const unsigned char* srcBgr, int width, int height, size_t srcStride, unsigned char* dstBgr, size_t dstStride) {
        return w2x_pool_submit(h_, srcBgr, width, height, srcStride, dstBgr, dstStride);
    }
    int submitResized(const unsigned char* srcBgr, int width, int height, size_t srcStride, unsigned char* dstBgr, int dstWidth, int dstHeight,
                      size_t dstStride) {
        return w2x_pool_submit_resized(h_, srcBgr, width, height, srcStride, dstBgr, dstWidth, dstHeight, dstStride);
    }
    int submitU16(const uint16_t* srcBgr, int width, int height, size_t srcStride, uint16_t* dstBgr, size_t dstStride) {
        return w2x_pool_submit_u16(h_, srcBgr, width, height, srcStride, dstBgr, dstStride);
    }
    bool wait(int ticket) { return w2x_pool_wait(h_, ticket) != 0; }
    // the pool's index-th engine (borrowed), e.g. for w2x_render_bgra
    w2x_engine* engine(int index) const { return w2x_pool_engine(h_, index); }
    void setMessageCallback(MessageCallback cb) {
        msg_ = std::move(cb);
        w2x_pool_set_message_callback(h_, msg_ ? &Img2ImgPool::onMessage : nullptr, this);
    }

private:
    static void onMessage(int sev, const char* m, void* self) { static_cast<Img2ImgPool*>(self)->msg_(static_cast<Severity>(sev), m); }
    w2x_pool* h_;
    MessageCallback msg_;
};

}  // namespace trt
