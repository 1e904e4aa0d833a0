// Header-only C++ mirror of the reference's public class over the C ABI (vstab.h).
//
// Same member names, defaults and exception types as class Stabilizer of
// /root/reference/include/stabilizer.hpp:106-475, so that callers shaped like
// /root/reference/src/main_utils.cpp:300-302, :371-395, :459-493 compile unchanged:
//     Stabilizer stabilizer(past, future, workingHeight);
//     stabilizer.setStabilizationMode(StabilizationMode::ACCUMULATED_FULL_LOCK);
//     out = stabilizer.stabilizeFrame(frame);
// cv::Mat is replaced by the POD ImageView (no OpenCV in this image); cv::Mat overloads are
// available under VSTAB_WITH_OPENCV.  All pixel work happens in libvstab.so on the GPU.
#pragma once

#include <cstddef>
#include <cstdint>
#include <stdexcept>
#include <string>
#include <vector>

#include "vstab.h"

#ifdef VSTAB_WITH_OPENCV
#include <opencv2/core.hpp>
#endif

// /root/reference/include/stabilizer.hpp:31-38
enum class StabilizationMode {
    ACCUMULATED_FULL_LOCK,
    ORB_FULL_LOCK,
    SIFT_FULL_LOCK,
    TRANSLATION_LOCK,
    ROTATION_LOCK,
    GLOBAL_SMOOTHING
};

// /root/reference/include/stabilizer.hpp:44-57 (cv::Vec2d -> double[2])
struct HomographyParameters {
    double s{1.0};
    double theta{0.0};
    double k{1.0};
    double delta{0.0};
    double t[2]{0.0, 0.0};
    double v[2]{0.0, 0.0};
};

// 8-bit BGR, HWC, `step` bytes per row: the fields of cv::Mat the reference relies on.
struct ImageView {
    uint8_t* data{nullptr};
    int rows{0};
    int cols{0};
    size_t step{0};
};

// A YUV 4:2:0 frame (NV12 / I420): base pointer and where its planes are (vstab_yuv_layout, e.g. from
// vstab_yuv_layout_packed for ffmpeg rawvideo, or offsets/steps of an NVDEC surface).
struct YuvView {
    uint8_t* data{nullptr};
    vstab_yuv_layout layout{};
    int rows{0};
    int cols{0};
};

// Owning image returned by stabilizeFrame (the reference returns a fresh cv::Mat).
struct Image {
    std::vector<uint8_t> pixels;
    int rows{0};
    int cols{0};
    size_t step{0};
    ImageView view() { return ImageView{pixels.data(), rows, cols, step}; }
};

class Stabilizer {
public:
    // Stabilizer(size_t pastFrames = 15, size_t futureFrames = 15, int workingHeight = 360)
    explicit Stabilizer(size_t pastFrames = 15, size_t futureFrames = 15, int workingHeight = 360, int device = 0)
        : totalPastFrames_(pastFrames), totalFutureFrames_(futureFrames) {
        vstab_status st = vstab_create(pastFrames, futureFrames, workingHeight, device, &h_);
        if (st == VSTAB_ERR_INVALID_ARGUMENT) throw std::invalid_argument(vstab_last_error(nullptr));
        if (st != VSTAB_OK) throw std::runtime_error(vstab_last_error(nullptr));
    }
    ~Stabilizer() { vstab_destroy(h_); }
    Stabilizer(const Stabilizer&) = delete;
    Stabilizer& operator=(const Stabilizer&) = delete;

    // cv::Mat stabilizeFrame(const cv::Mat& frame)
    Image stabilizeFrame(const ImageView& frame) {
        Image out;
        out.rows = frame.rows;
        out.cols = frame.cols;
        out.step = static_cast<size_t>(frame.cols) * 3;
        out.pixels.resize(out.step * static_cast<size_t>(frame.rows > 0 ? frame.rows : 0));
        stabilizeFrame(frame, out.view());
        return out;
    }
    // Same, into a caller-owned buffer (e.g. pinned memory from vstab_host_alloc).
    void stabilizeFrame(const ImageView& frame, const ImageView& out) {
        check(vstab_stabilize_frame(h_, frame.data, frame.rows, frame.cols, frame.step, out.data, out.step));
    }

    // stabilizeFrame on YUV frames: `in` is converted to BGR on the device, the BGR output to `out`'s format before it leaves
    // (out == BGR2YUV_I420(stabilizeFrame(YUV2BGR(in))), see vstab.h).  Throws like stabilizeFrame.
    void stabilizeFrameYuv(const YuvView& in, const YuvView& out) {
        if (out.rows != in.rows || out.cols != in.cols) throw std::invalid_argument("stabilizeFrameYuv: output size differs from input size");
        check(vstab_stabilize_frame_yuv(h_, in.data, &in.layout, in.rows, in.cols, out.data, &out.layout));
    }

#ifdef VSTAB_WITH_OPENCV
    cv::Mat stabilizeFrame(const cv::Mat& frame) {
        cv::Mat out(frame.rows, frame.cols, CV_8UC3);
        check(vstab_stabilize_frame(h_, frame.data, frame.rows, frame.cols, frame.step, out.data, out.step));
        return out;
    }
#endif

    void setStabilizationMode(StabilizationMode mode) { check(vstab_set_mode(h_, static_cast<int>(mode))); }

    // The reference selects its feathered-trail output (copyFeathered, src/stabilizer.cpp:1303-1307) at compile time with
    // `#if 0`; here it is a run-time switch, off by default.
    void setTrailCompositing(bool enable) { check(vstab_set_trail(h_, enable ? 1 : 0)); }
    // Auto-crop (vstab_set_crop, include/vstab.h): zoom each output just enough to hide its border, up to maxZoom
    // (1 < maxZoom <= 4; 1 turns it off), the zoom falling back by at most `release` per call.  Beyond the reference.
    void setAutoCrop(double maxZoom, double release = 0.002) { check(vstab_set_crop(h_, maxZoom, release)); }

    // TRANSLATION_LOCK / ROTATION_LOCK evaluate to the identity in the reference (include/stabilizer.hpp:23 "@todo fix
    // partial locking modes"); with this switch its formulas (src/stabilizer.cpp:1246-1260) are fed with the accumulated
    // lock, which is what they were written for.  Off by default.
    void setPartialLockFix(bool enable) { check(vstab_set_partial_lock_fix(h_, enable ? 1 : 0)); }

    inline size_t totalFrameWindowSize() const { return totalPastFrames_ + 1 + totalFutureFrames_; }

    // static bool decomposeHomography(const cv::Mat& H, HomographyParameters&, cv::Point2d rot_center = {0,0})
    static bool decomposeHomography(const double H[9], HomographyParameters& params_out, double cx = 0.0, double cy = 0.0) {
        vstab_hparams p;
        int r = vstab_decompose_homography(H, cx, cy, &p);
        if (r < 0) throw std::invalid_argument("Error: Input homography matrix must be a non-empty 3x3 CV_64F matrix.");
        if (r == 0) return false;
        params_out.s = p.s; params_out.theta = p.theta; params_out.k = p.k; params_out.delta = p.delta;
        params_out.t[0] = p.t[0]; params_out.t[1] = p.t[1]; params_out.v[0] = p.v[0]; params_out.v[1] = p.v[1];
        return true;
    }

    // static cv::Mat composeHomography(const HomographyParameters&, cv::Point2d rot_center = {0,0})
    static void composeHomography(const HomographyParameters& params, double H_out[9], double cx = 0.0, double cy = 0.0) {
        vstab_hparams p;
        p.s = params.s; p.theta = params.theta; p.k = params.k; p.delta = params.delta;
        p.t[0] = params.t[0]; p.t[1] = params.t[1]; p.v[0] = params.v[0]; p.v[1] = params.v[1];
        vstab_compose_homography(&p, cx, cy, H_out);
    }

    vstab_t* handle() { return h_; }

private:
    void check(vstab_status st) {
        if (st == VSTAB_OK) return;
        const std::string msg = vstab_last_error(h_);
        if (st == VSTAB_ERR_INVALID_ARGUMENT || st == VSTAB_ERR_SIZE_CHANGED) throw std::invalid_argument(msg);
        if (st == VSTAB_ERR_STATE) throw std::logic_error(msg);        // the reference asserts here
        throw std::runtime_error(msg);
    }

    vstab_t* h_{nullptr};
    size_t totalPastFrames_{0};
    size_t totalFutureFrames_{0};
};
