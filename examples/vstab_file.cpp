// Headless file front end over include/stabilizer.hpp: the reference's main loop for --file input
// (/root/reference/src/main.cpp:196-236, src/main_utils.cpp:397-417 captureFrame, :459-493
// processAndDisplayFrames) without the GUI: frames come from a raw BGR24 stream (what
// `ffmpeg -f rawvideo -pix_fmt bgr24` writes) instead of cv::VideoCapture, the stabilized frames go
// to a raw BGR24 stream instead of imshow.  --pix-fmt nv12|yuv420p reads (and, unless --out-pix-fmt says otherwise, writes)
// raw 4:2:0 frames instead, what decoders produce (`ffmpeg -f rawvideo -pix_fmt yuv420p`): they are converted on the GPU, so
// half the bytes per frame cross the host link.  Flags follow the reference's CLI
// (src/main_utils.cpp:35-236: --file, --past-window, --future-window, --working-height); the
// stabilization-mode keys of handleStabilizationControls (:371-395) become --mode / --mode-at.
//
//   vstab_file --file in.bgr --width 1920 --height 1080 --out out.bgr
//              [--past-window 60] [--future-window 45] [--working-height 360]
//              [--mode global|lock|orb|sift|translation|rotation] [--mode-at CALL] [--side-by-side] [--frames N]
//              [--pix-fmt bgr24|nv12|yuv420p] [--out-pix-fmt bgr24|nv12|yuv420p]
//
// --side-by-side writes [delayed original | stabilized] (2*width columns): the original is delayed by
// `future-window` frames through the same deque the reference keeps (originalFrameBuffer, :466-472), so both halves
// show the same source frame; nothing is written while that buffer fills (the reference prints "Buffering frames").
// "-" means stdin / stdout.  Exit status: 0 ok, 1 bad usage, 2 I/O, 3 stabilizer error.
#include <chrono>
#include <cstdio>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <string>
#include <vector>

#include "stabilizer.hpp"

namespace {

struct Options {
    std::string in, out = "-";
    int width = 0, height = 0;
    long frames = -1, mode_at = 0;
    long past = -1, future = -1;         // default: 2.0 s / 1.5 s at 30 fps (src/main.cpp:205-206)
    int working_height = 360;            // src/main_utils.hpp:27
    bool side_by_side = false, have_mode = false;
    StabilizationMode mode = StabilizationMode::GLOBAL_SMOOTHING;
    int pix_fmt = 0, out_pix_fmt = -1;   // 0 = bgr24, else vstab_pixel_format; -1: as the input
    double crop = 1.0, crop_release = 0.002;   // auto-crop (1: off)
};

// ffmpeg's pixel format names
bool parse_pix_fmt(const std::string& s, int& f) {
    if (s == "bgr24") f = 0;
    else if (s == "nv12") f = VSTAB_PIX_NV12;
    else if (s == "yuv420p") f = VSTAB_PIX_I420;
    else return false;
    return true;
}

bool parse_mode(const std::string& s, StabilizationMode& m) {
    if (s == "global") m = StabilizationMode::GLOBAL_SMOOTHING;
    else if (s == "lock") m = StabilizationMode::ACCUMULATED_FULL_LOCK;
    else if (s == "orb") m = StabilizationMode::ORB_FULL_LOCK;
    else if (s == "sift") m = StabilizationMode::SIFT_FULL_LOCK;
    else if (s == "translation") m = StabilizationMode::TRANSLATION_LOCK;
    else if (s == "rotation") m = StabilizationMode::ROTATION_LOCK;
    else return false;
    return true;
}

// --crop MAX_ZOOM[,RELEASE]: 1 < MAX_ZOOM <= 4, RELEASE > 0 (default 0.002 per call), ceil((MAX_ZOOM - 1) / RELEASE) <= 4096
bool parse_crop(const std::string& s, double& max_zoom, double& release) {
    const size_t comma = s.find(',');
    const std::string a = s.substr(0, comma), b = comma == std::string::npos ? "" : s.substr(comma + 1);
    if (a.empty() || (comma != std::string::npos && b.empty())) return false;
    char* end = nullptr;
    max_zoom = std::strtod(a.c_str(), &end);
    if (*end) return false;
    release = 0.002;
    if (!b.empty()) { release = std::strtod(b.c_str(), &end); if (*end) return false; }
    return max_zoom > 1.0 && max_zoom <= 4.0 && release > 0.0 && std::isfinite(release) &&
           std::ceil((max_zoom - 1.0) / release) <= 4096.0;
}

int usage(const char* argv0) {
    std::fprintf(stderr,
                 "usage: %s --file <in.bgr|-> --width W --height H [--out <out.bgr|->] [--past-window N] [--future-window N]\n"
                 "          [--working-height N] [--mode global|lock|orb|sift|translation|rotation] [--mode-at CALL]\n"
                 "          [--side-by-side] [--frames N] [--pix-fmt bgr24|nv12|yuv420p] [--out-pix-fmt bgr24|nv12|yuv420p]\n"
                 "          [--crop MAX_ZOOM[,RELEASE]]\n", argv0);
    return 1;
}

bool read_full(std::FILE* f, uint8_t* p, size_t n) {
    while (n) {
        const size_t r = std::fread(p, 1, n, f);
        if (r == 0) return false;
        p += r; n -= r;
    }
    return true;
}

}  // namespace

int main(int argc, char** argv) {
    Options o;
    for (int i = 1; i < argc; ++i) {
        const std::string a = argv[i];
        auto next = [&](const char* what) -> const char* {
            if (i + 1 >= argc) { std::fprintf(stderr, "Error: %s requires a value.\n", what); std::exit(1); }
            return argv[++i];
        };
        if (a == "--help" || a == "-h") return usage(argv[0]);
        else if (a == "--file") o.in = next("--file");
        else if (a == "--out") o.out = next("--out");
        else if (a == "--width") o.width = std::atoi(next("--width"));
        else if (a == "--height") o.height = std::atoi(next("--height"));
        else if (a == "--frames") o.frames = std::atol(next("--frames"));
        else if (a == "--past-window") o.past = std::atol(next("--past-window"));
        else if (a == "--future-window") o.future = std::atol(next("--future-window"));
        else if (a == "--working-height") o.working_height = std::atoi(next("--working-height"));
        else if (a == "--mode") { if (!parse_mode(next("--mode"), o.mode)) return usage(argv[0]); o.have_mode = true; }
        else if (a == "--mode-at") o.mode_at = std::atol(next("--mode-at"));
        else if (a == "--side-by-side") o.side_by_side = true;
        else if (a == "--crop") { if (!parse_crop(next("--crop"), o.crop, o.crop_release)) return usage(argv[0]); }
        else if (a == "--pix-fmt") { if (!parse_pix_fmt(next("--pix-fmt"), o.pix_fmt)) return usage(argv[0]); }
        else if (a == "--out-pix-fmt") { if (!parse_pix_fmt(next("--out-pix-fmt"), o.out_pix_fmt)) return usage(argv[0]); }
        else { std::fprintf(stderr, "Error: unknown argument %s\n", a.c_str()); return usage(argv[0]); }
    }
    if (o.in.empty() || o.width <= 0 || o.height <= 0) return usage(argv[0]);
    if (o.out_pix_fmt < 0) o.out_pix_fmt = o.pix_fmt;
    // 4:2:0 frames: the packed rawvideo layouts (even sizes only); the side-by-side view is a BGR picture
    vstab_yuv_layout lin{}, lout{};
    const bool yuv = o.pix_fmt || o.out_pix_fmt;
    if (yuv && o.side_by_side) { std::fprintf(stderr, "Error: --side-by-side needs bgr24 input and output.\n"); return 1; }
    const size_t bgr_bytes = (size_t)o.width * 3 * (size_t)o.height;
    const size_t in_bytes = o.pix_fmt ? vstab_yuv_layout_packed(o.pix_fmt, o.height, o.width, &lin) : bgr_bytes;
    const size_t out_bytes = o.out_pix_fmt ? vstab_yuv_layout_packed(o.out_pix_fmt, o.height, o.width, &lout) : bgr_bytes;
    if (!in_bytes || !out_bytes) { std::fprintf(stderr, "Error: 4:2:0 frames need an even width and height.\n"); return 1; }
    if (yuv && (!o.pix_fmt || !o.out_pix_fmt)) {          // the YUV calls take 4:2:0 on both sides (NV12 / I420 in any mix)
        std::fprintf(stderr, "Error: --pix-fmt and --out-pix-fmt must both be bgr24 or both be 4:2:0.\n");
        return 1;
    }
    const double fps = 30.0;
    if (o.past < 0) o.past = (long)(2.0 * fps);
    if (o.future < 0) o.future = (long)(1.5 * fps);

    std::FILE* fin = o.in == "-" ? stdin : std::fopen(o.in.c_str(), "rb");
    std::FILE* fout = o.out == "-" ? stdout : std::fopen(o.out.c_str(), "wb");
    if (!fin || !fout) { std::fprintf(stderr, "Error: cannot open %s\n", !fin ? o.in.c_str() : o.out.c_str()); return 2; }

    const size_t step = (size_t)o.width * 3;
    uint8_t *hin = nullptr, *hout = nullptr;
    std::deque<std::vector<uint8_t>> originalFrameBuffer;       // src/main_utils.cpp:466
    std::vector<uint8_t> row;
    if (o.side_by_side) row.resize(2 * step);
    long n = 0, written = 0;
    int rc = 0;
    try {
        Stabilizer stabilizer((size_t)o.past, (size_t)o.future, o.working_height);   // argument errors throw before any device work
        if (o.crop > 1.0) stabilizer.setAutoCrop(o.crop, o.crop_release);
        // pinned staging buffers: the per-frame call copies straight from / into them
        hin = static_cast<uint8_t*>(vstab_host_alloc(in_bytes));
        hout = static_cast<uint8_t*>(vstab_host_alloc(out_bytes));
        if (!hin || !hout) throw std::runtime_error("pinned host allocation failed");
        const auto t0 = std::chrono::steady_clock::now();
        while ((o.frames < 0 || n < o.frames) && read_full(fin, hin, in_bytes)) {
            if (o.have_mode && n == o.mode_at) stabilizer.setStabilizationMode(o.mode);
            if (yuv)
                stabilizer.stabilizeFrameYuv(YuvView{hin, lin, o.height, o.width}, YuvView{hout, lout, o.height, o.width});
            else
                stabilizer.stabilizeFrame(ImageView{hin, o.height, o.width, step}, ImageView{hout, o.height, o.width, step});
            ++n;
            if (!o.side_by_side) {
                if (std::fwrite(hout, 1, out_bytes, fout) != out_bytes) { rc = 2; break; }
                ++written;
                continue;
            }
            originalFrameBuffer.emplace_back(hin, hin + in_bytes);
            if (originalFrameBuffer.size() > (size_t)o.future) {
                const std::vector<uint8_t>& delayed = originalFrameBuffer.front();
                for (int y = 0; y < o.height && rc == 0; ++y) {
                    std::memcpy(row.data(), delayed.data() + (size_t)y * step, step);
                    std::memcpy(row.data() + step, hout + (size_t)y * step, step);
                    if (std::fwrite(row.data(), 1, row.size(), fout) != row.size()) rc = 2;
                }
                originalFrameBuffer.pop_front();
                ++written;
                if (rc) break;
            }
        }
        const double sec = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        std::fprintf(stderr, "%ld frames in, %ld frames out, %.1f frames/s (window %zu)\n", n, written,
                     sec > 0 ? n / sec : 0.0, stabilizer.totalFrameWindowSize());
    } catch (const std::invalid_argument& e) {
        std::fprintf(stderr, "Error: %s\n", e.what());
        rc = 1;
    } catch (const std::exception& e) {
        std::fprintf(stderr, "Error: %s\n", e.what());
        rc = 3;
    }
    if (hin) vstab_host_free(hin);
    if (hout) vstab_host_free(hout);
    if (fin != stdin) std::fclose(fin);
    if (fout != stdout) std::fclose(fout); else std::fflush(stdout);
    return rc;
}
