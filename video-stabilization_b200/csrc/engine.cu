// Host side of the C ABI (include/vstab.h): the streaming Stabilizer instance, the offline
// (frame-sharded) runner and the single-kernel test entry points.  This file only
// orchestrates: all arithmetic of the hot path runs in the kernels of this directory,
// there is no CPU fallback (every entry point needs a CUDA device).
//
// Streaming state mirrors class Stabilizer (/root/reference/include/stabilizer.hpp:430-474)
// but lives in device memory: a ring of W = past+1+future full-resolution frames (the
// reference's deque of cloned cv::Mat, :437), the per-slot channel sums, two gray pyramids
// (prevGray_/gray, :439), the corner list (prevPoints_, :440), a ring of 3x3 transforms
// and the accumulated transform (:444).  The host keeps only integer indices, so a call
// enqueues kernels and copies without ever reading a result back except the output frame.
#include <atomic>
#include <dlfcn.h>
#include <memory>
#include <mutex>
#include <utility>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <cstdio>
#include <cstring>
#include <new>
#include <optional>
#include <string>
#include <vector>

#include "../../include/vstab.h"
#include "homography.cuh"
#include "kernels.h"

using namespace vstabk;

namespace vstabk {
static std::atomic<long long> g_launches{0};
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
long long launch_count() { return g_launches.load(std::memory_order_relaxed); }
int device_sm_count() {
    static std::atomic<int> cache[64];
    int dev = 0;
    cudaGetDevice(&dev);
    int n = cache[dev & 63].load(std::memory_order_relaxed);
    if (n <= 0) {
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) { cudaGetLastError(); n = 148; }
        cache[dev & 63].store(n, std::memory_order_relaxed);
    }
    return n;
}
GraphCache::~GraphCache() {
    for (auto& e : entries) {
        if (e.exec) cudaGraphExecDestroy(e.exec);
        if (e.graph) cudaGraphDestroy(e.graph);
    }
}
}  // namespace vstabk

namespace {

// Per-stage device timing with CUDA events on the instance stream (bench.py's roofline numbers).
enum Stage { ST_INGEST = 0, ST_PYRAMID, ST_GFTT, ST_LK, ST_FIT, ST_SMOOTH, ST_WARP, ST_ACC, ST_COUNT };
struct StageTimer {
    bool enabled = false;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ev[ST_COUNT];
    void begin(int s, cudaStream_t q) {
        if (!enabled) return;
        cudaEvent_t a, b;
        cudaEventCreate(&a); cudaEventCreate(&b);
        ev[s].push_back({a, b});
        cudaEventRecord(a, q);
    }
    void end(int s, cudaStream_t q) { if (enabled) cudaEventRecord(ev[s].back().second, q); }
    // sums and clears; returns launches (event pairs) per stage in counts
    void collect(float* ms, int* counts) {
        for (int s = 0; s < ST_COUNT; ++s) {
            float tot = 0.f;
            for (auto& pr : ev[s]) {
                float t = 0.f;
                cudaEventSynchronize(pr.second);
                cudaEventElapsedTime(&t, pr.first, pr.second);
                tot += t;
                cudaEventDestroy(pr.first); cudaEventDestroy(pr.second);
            }
            ms[s] = tot; counts[s] = (int)ev[s].size();
            ev[s].clear();
        }
    }
    ~StageTimer() { float m[ST_COUNT]; int c[ST_COUNT]; collect(m, c); }
};

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

#define CK(call)                                                                          \
    do {                                                                                  \
        cudaError_t e__ = (call);                                                         \
        if (e__ != cudaSuccess) {                                                         \
            set_err(std::string(#call) + ": " + cudaGetErrorString(e__));                 \
            return VSTAB_ERR_CUDA;                                                        \
        }                                                                                 \
    } while (0)

thread_local std::string g_err;   // for entry points without an instance
// a SIFT matcher launch (launch_l2_match / launch_l2_nn_batch) returned false
constexpr const char* kL2MapErr = "SIFT matcher: cuTensorMapEncodeTiled (the driver's tensor-map encoder) is missing or rejected the descriptor arrays";
void nccl_comm_destroy(void* comm);

// auto-crop parameters (vstab_set_crop / vstab_offline_set_crop); max_zoom == 1 turns the crop off
constexpr int kCropMaxR = 4096;
bool crop_params(double max_zoom, double release, CropArgs* out, std::string& err) {
    CropArgs c{1.0, 0.0, 0};
    if (max_zoom != 1.0) {
        if (!(max_zoom > 1.0 && max_zoom <= 4.0) || !(release > 0.0) || !std::isfinite(release)) {
            err = "auto-crop: max_zoom must be 1 (off) or in (1, 4], and release a finite value > 0";
            return false;
        }
        const double R = std::ceil((max_zoom - 1.0) / release);
        if (!(R <= kCropMaxR)) { err = "auto-crop: (max_zoom - 1) / release exceeds 4096 calls"; return false; }
        c.max_zoom = max_zoom; c.release = release; c.R = (int)R;
    }
    *out = c;
    return true;
}

// VSTAB_GUARD=1 (tests): every device buffer of the library is allocated between two 4 KB guard bands filled with a pattern;
// when the buffer is released the bands are read back and every byte that changed counts as an out-of-bounds WRITE
// (vstab_debug_guard_violations).  compute-sanitizer is closed on the GPU pool this was developed on; this is the bounds
// check "of your own" that runs in its place over the whole GPU test suite (tests/conftest.py).
constexpr size_t kGuardBytes = 4096;
std::atomic<long long> g_guard_violations{0};
std::atomic<long long> g_guard_buffers{0};
inline bool guard_enabled() {
    static const bool on = getenv("VSTAB_GUARD") && atoi(getenv("VSTAB_GUARD")) != 0;
    return on;
}

struct DevBuf {
    void* p = nullptr;
    size_t guarded_bytes = 0;               // > 0: p sits kGuardBytes into an allocation of guarded_bytes + 2 * kGuardBytes
    ~DevBuf() { release(); }
    void release() {
        if (!p) return;
        if (guarded_bytes) {
            unsigned char* base = (unsigned char*)p - kGuardBytes;
            std::vector<unsigned char> g(2 * kGuardBytes);
            if (cudaMemcpy(g.data(), base, kGuardBytes, cudaMemcpyDeviceToHost) == cudaSuccess &&
                cudaMemcpy(g.data() + kGuardBytes, (unsigned char*)p + guarded_bytes, kGuardBytes, cudaMemcpyDeviceToHost) == cudaSuccess) {
                long long bad = 0;
                for (unsigned char c : g) bad += c != 0xA5;
                if (bad) {
                    g_guard_violations.fetch_add(bad);
                    fprintf(stderr, "[vstab guard] %lld byte(s) written outside a %zu-byte device buffer\n", bad, guarded_bytes);
                }
            } else {
                cudaGetLastError();
            }
            cudaFree(base);
        } else {
            cudaFree(p);
        }
        p = nullptr; guarded_bytes = 0;
    }
    cudaError_t alloc(size_t bytes) {
        release();
        if (!bytes) bytes = 1;
        if (!guard_enabled()) return cudaMalloc(&p, bytes);
        const size_t padded = (bytes + 255) & ~(size_t)255;        // keep the tail band's start aligned; slack bytes are guard too
        void* base = nullptr;
        cudaError_t e = cudaMalloc(&base, padded + 2 * kGuardBytes);
        if (e != cudaSuccess) return e;
        cudaMemset(base, 0xA5, kGuardBytes);
        cudaMemset((unsigned char*)base + kGuardBytes + bytes, 0xA5, padded - bytes + kGuardBytes);
        p = (unsigned char*)base + kGuardBytes;
        guarded_bytes = bytes;
        g_guard_buffers.fetch_add(1);
        return cudaSuccess;
    }
    template <typename T> T* as() const { return (T*)p; }
};

// Everything that depends only on (rows, cols, working height) and a frame-batch capacity.
struct Geometry {
    int rows = 0, cols = 0, wh = 0, ww = 0;
    double scale = 1.0;
    size_t pitch = 0, frame_bytes = 0;
    PyrDesc pd{};
    IngestPlan plan{};
    DevBuf xtab, ytab;
    DevBuf nn_x, nn_y;           // cv::resize INTER_NEAREST offsets of the ORB / SIFT conditioning (nn_tables)
    bool nn_ready = false;
    int min_distance = 0;

    vstab_status init(int r, int c, int working_height, std::string& err) {
        rows = r; cols = c; wh = working_height;
        scale = (double)working_height / (double)r;                     // stabilizer.cpp:117
        ww = (int)(c * scale);                                         // stabilizer.cpp:118
        if (ww < 8 || wh < 8) { err = "working size too small"; return VSTAB_ERR_INVALID_ARGUMENT; }
        pitch = align_up((size_t)c * 3, 16);
        frame_bytes = align_up(pitch * (size_t)r, 256);
        pd = make_pyr_desc(ww, wh);
        plan.src_w = c; plan.src_h = r; plan.dst_w = ww; plan.dst_h = wh;
        plan.mode = (ww == c && wh == r) ? 0 : ((c == 2 * ww && r == 2 * wh) ? 1 : 2);
        // destination rows per CTA.  Measured on B200, 1080p -> 360 (3 source rows per destination row), ms per 256 frames:
        // 1 row 0.51, 2 0.43, 3-4 0.41, 8 0.45; 4K -> 360 (6 source rows per destination row): 2 rows 85 % of the HBM roofline,
        // 4 rows 76 % -- so about 12 source rows per CTA.
        plan.rows_per_band = wh >= 360 ? ((long)r >= 5L * wh ? 2 : 4) : 1;
        plan.nbands = (wh + plan.rows_per_band - 1) / plan.rows_per_band;
        std::vector<int4> hx(ww), hy(wh);
        build_ingest_tables(c, ww, plan.mode, hx.data());
        build_ingest_tables(r, wh, plan.mode, hy.data());
        if (xtab.alloc(sizeof(int4) * ww) != cudaSuccess || ytab.alloc(sizeof(int4) * wh) != cudaSuccess) {
            err = "cudaMalloc(ingest tables) failed"; return VSTAB_ERR_CUDA;
        }
        if (cudaMemcpy(xtab.p, hx.data(), sizeof(int4) * ww, cudaMemcpyHostToDevice) != cudaSuccess ||
            cudaMemcpy(ytab.p, hy.data(), sizeof(int4) * wh, cudaMemcpyHostToDevice) != cudaSuccess) {
            err = "cudaMemcpy(ingest tables) failed"; return VSTAB_ERR_CUDA;
        }
        plan.xtab = xtab.as<int4>();
        plan.ytab = ytab.as<int4>();
        min_distance = (int)(10 * ((double)wh / 720.0));                // stabilizer.cpp:938-940
        return VSTAB_OK;
    }

    // nn_x / nn_y, built on first use: only the ORB / SIFT paths condition frames
    cudaError_t nn_tables() {
        if (nn_ready) return cudaSuccess;
        auto table = [](DevBuf& t, int src, int dst) {
            std::vector<int> h(dst);
            build_nn_table(src, dst, h.data());
            const cudaError_t e = t.alloc(sizeof(int) * dst);
            return e != cudaSuccess ? e : cudaMemcpy(t.p, h.data(), sizeof(int) * dst, cudaMemcpyHostToDevice);
        };
        cudaError_t e = table(nn_x, cols, ww);
        if (e == cudaSuccess) e = table(nn_y, rows, wh);
        nn_ready = e == cudaSuccess;
        return e;
    }
};

bool device_ok(int device, std::string& err) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) {
        err = std::string("no CUDA device: ") + cudaGetErrorString(e) + " (this library has no CPU fallback)";
        return false;
    }
    if (device < 0 || device >= n) { err = "bad device index"; return false; }
    cudaDeviceProp p;
    if (cudaGetDeviceProperties(&p, device) != cudaSuccess) { err = "cudaGetDeviceProperties failed"; return false; }
    if (p.major < 10) {
        err = "device is sm_" + std::to_string(p.major * 10 + p.minor) + "; kernels are built for sm_100a only";
        return false;
    }
    if (cudaSetDevice(device) != cudaSuccess) { err = "cudaSetDevice failed"; return false; }
    return true;
}

// ---- YUV 4:2:0 frames (vstab_yuv_layout): plane geometry, checks, device staging, plane copies -------------------------
inline int yuv_nplanes(int fmt) { return fmt == VSTAB_PIX_NV12 ? 2 : 3; }
inline size_t yuv_row_bytes(int fmt, int k, int cols) { return k == 0 || fmt == VSTAB_PIX_NV12 ? (size_t)cols : (size_t)cols / 2; }
inline int yuv_rows(int k, int rows) { return k == 0 ? rows : rows / 2; }

// end of the last plane byte of a frame laid out as *L, or 0 (and `err`) when the layout does not describe a rows x cols frame
size_t yuv_extent(const vstab_yuv_layout* L, int rows, int cols, std::string& err) {
    if (!L) { err = "null YUV layout"; return 0; }
    if (L->format != VSTAB_PIX_NV12 && L->format != VSTAB_PIX_I420) { err = "unknown pixel format " + std::to_string(L->format); return 0; }
    if (rows < 2 || cols < 2 || (rows & 1) || (cols & 1)) {
        err = "YUV 4:2:0 frames need even rows and cols. Rows: " + std::to_string(rows) + ", Cols: " + std::to_string(cols);
        return 0;
    }
    size_t end = 0;
    for (int k = 0; k < yuv_nplanes(L->format); ++k) {
        const size_t rb = yuv_row_bytes(L->format, k, cols);
        if (L->step[k] < rb) { err = "row step of YUV plane " + std::to_string(k) + " smaller than its " + std::to_string(rb) + " bytes"; return 0; }
        const size_t e = L->offset[k] + L->step[k] * (size_t)(yuv_rows(k, rows) - 1) + rb;
        if (e > end) end = e;
    }
    return end;
}

size_t yuv_packed(int fmt, int rows, int cols, vstab_yuv_layout* out) {
    const size_t y = (size_t)rows * cols, c = y / 4;
    *out = vstab_yuv_layout{};
    out->format = fmt;
    out->step[0] = (size_t)cols;
    out->offset[1] = y;
    if (fmt == VSTAB_PIX_NV12) {
        out->step[1] = (size_t)cols;
    } else {
        out->step[1] = out->step[2] = (size_t)cols / 2;
        out->offset[2] = y + c;
    }
    return y + 2 * c;
}

// Layout of the library's own YUV staging buffers: the packed one when cols % 8 == 0 (then every plane and frame offset is a
// multiple of 8 and the conversions take their word paths; 1080p, 4K), otherwise rows padded to 16 bytes.
vstab_yuv_layout yuv_staging_layout(int fmt, int rows, int cols, size_t* frame_bytes) {
    vstab_yuv_layout L;
    size_t bytes = yuv_packed(fmt, rows, cols, &L);
    if (cols % 8) {
        size_t off = 0;
        for (int k = 0; k < yuv_nplanes(fmt); ++k) {
            L.offset[k] = off;
            L.step[k] = align_up(yuv_row_bytes(fmt, k, cols), 16);
            off += L.step[k] * (size_t)yuv_rows(k, rows);
        }
        bytes = off;
    }
    *frame_bytes = bytes;
    return L;
}

size_t yuv_staging_bytes(int rows, int cols) {            // one frame, either format
    size_t a = 0, b = 0;
    yuv_staging_layout(VSTAB_PIX_NV12, rows, cols, &a);
    yuv_staging_layout(VSTAB_PIX_I420, rows, cols, &b);
    return a > b ? a : b;
}

YuvPlanes yuv_planes_of(const vstab_yuv_layout& L) {
    YuvPlanes p{};
    p.off_y = L.offset[0]; p.step_y = L.step[0];
    p.off_u = L.offset[1]; p.step_u = L.step[1];
    if (L.format == VSTAB_PIX_NV12) { p.off_v = L.offset[1] + 1; p.step_v = L.step[1]; p.cstep = 2; }
    else { p.off_v = L.offset[2]; p.step_v = L.step[2]; p.cstep = 1; }
    return p;
}

bool same_planes(const vstab_yuv_layout& a, const vstab_yuv_layout& b) {
    if (a.format != b.format) return false;
    for (int k = 0; k < yuv_nplanes(a.format); ++k)
        if (a.offset[k] != b.offset[k] || a.step[k] != b.step[k]) return false;
    return true;
}

// n frames between two layouts of the same format, one cudaMemcpy2DAsync per plane and frame -- or ONE copy when both sides
// are tightly packed rawvideo (no bytes between planes or frames that the copy could clobber)
cudaError_t yuv_copy(uint8_t* dst, const vstab_yuv_layout& dl, size_t dst_fs, const uint8_t* src, const vstab_yuv_layout& sl,
                     size_t src_fs, long n, int rows, int cols, cudaMemcpyKind kind, cudaStream_t q) {
    vstab_yuv_layout P;
    const size_t packed = yuv_packed(dl.format, rows, cols, &P);
    if (same_planes(dl, P) && same_planes(sl, P) && (n == 1 || (dst_fs == packed && src_fs == packed)))
        return cudaMemcpyAsync(dst, src, packed * (size_t)n, kind, q);
    for (long i = 0; i < n; ++i)
        for (int k = 0; k < yuv_nplanes(dl.format); ++k) {
            const cudaError_t e = cudaMemcpy2DAsync(dst + (size_t)i * dst_fs + dl.offset[k], dl.step[k], src + (size_t)i * src_fs + sl.offset[k],
                                                    sl.step[k], yuv_row_bytes(dl.format, k, cols), yuv_rows(k, rows), kind, q);
            if (e != cudaSuccess) return e;
        }
    return cudaSuccess;
}

// n BGR frames between two pitched layouts, one cudaMemcpy2DAsync per frame -- or ONE copy when neither side has a byte
// between rows or frames (the rule of yuv_copy)
cudaError_t bgr_copy(uint8_t* dst, size_t dst_step, size_t dst_fs, const uint8_t* src, size_t src_step, size_t src_fs, long n,
                     int rows, int cols, cudaMemcpyKind kind, cudaStream_t q) {
    const size_t rb = (size_t)cols * 3, packed = rb * (size_t)rows;
    if (dst_step == rb && src_step == rb && (n == 1 || (dst_fs == packed && src_fs == packed)))
        return cudaMemcpyAsync(dst, src, packed * (size_t)n, kind, q);
    for (long i = 0; i < n; ++i) {
        const cudaError_t e = cudaMemcpy2DAsync(dst + (size_t)i * dst_fs, dst_step, src + (size_t)i * src_fs, src_step, rb, rows, kind, q);
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

// ---- caller frames <-> the library's BGR frames (g.pitch bytes per row, g.frame_bytes per frame) ------------------------
// Every entry point moves its caller's frames in and out through the functions below.  Each direction has two phases, so
// that the copy and the conversion can run on different streams: input = transfer (BGR straight into the library's frames,
// host YUV into a staging buffer in the library's plane layout) then convert (YUV -> BGR); output = convert (BGR -> YUV, into
// staging for host memory, into the caller's frames for device memory) then transfer.  Device YUV frames are converted
// where they are.  Copies never touch the caller's bytes between rows, planes or frames.
struct FrameFmt {
    bool host = true;                          // host memory, else device memory
    const vstab_yuv_layout* yuv = nullptr;     // YUV 4:2:0 planes; null: BGR rows `step` bytes apart
    size_t step = 0;
    size_t stride = 0;                         // bytes from one frame of a run to the next

    // device BGR: the library reads and writes these frames where they are
    bool direct() const { return !host && !yuv; }
    // device bytes per frame of the staging buffer the transfer goes through (host YUV only), enough for either YUV format
    size_t staging_bytes(const Geometry& g) const { return host && yuv ? yuv_staging_bytes(g.rows, g.cols) : 0; }
    // `runs`: frames of a run sit `stride` bytes apart and must not overlap
    vstab_status check(int rows, int cols, bool runs, std::string& err, const char* step_err = "row step smaller than 3*cols") const {
        if (!yuv) {
            if (step >= (size_t)cols * 3) return VSTAB_OK;
            err = step_err;
            return VSTAB_ERR_INVALID_ARGUMENT;
        }
        const size_t extent = yuv_extent(yuv, rows, cols, err);
        if (!extent) return VSTAB_ERR_INVALID_ARGUMENT;
        if (runs && stride < extent) { err = "frame stride smaller than the extent of the YUV layout's planes"; return VSTAB_ERR_INVALID_ARGUMENT; }
        return VSTAB_OK;
    }
    // the staging frames of a host YUV format: the library's plane layout, `*fs` bytes apart
    vstab_yuv_layout staging(const Geometry& g, size_t* fs) const { return yuv_staging_layout(yuv->format, g.rows, g.cols, fs); }
};

// input, transfer: n caller frames at `src` -> BGR frames at `dst` (BGR), or -> `stage` (host YUV)
cudaError_t frames_in_transfer(const Geometry& g, const FrameFmt& f, const uint8_t* src, long n, uint8_t* dst, uint8_t* stage,
                               cudaStream_t q) {
    if (!f.yuv)
        return bgr_copy(dst, g.pitch, g.frame_bytes, src, f.step, f.stride, n, g.rows, g.cols,
                        f.host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, q);
    if (!f.host) return cudaSuccess;
    size_t sfs = 0;
    const vstab_yuv_layout S = f.staging(g, &sfs);
    return yuv_copy(stage, S, sfs, src, *f.yuv, f.stride, n, g.rows, g.cols, cudaMemcpyHostToDevice, q);
}

// input, convert: YUV -> BGR frames at `dst`, from `stage` (host) or from the caller's frames at `src` (device)
cudaError_t frames_in_convert(const Geometry& g, const FrameFmt& f, const uint8_t* src, long n, uint8_t* dst, const uint8_t* stage,
                              cudaStream_t q) {
    if (!f.yuv) return cudaSuccess;
    if (f.host) {
        size_t sfs = 0;
        const vstab_yuv_layout S = f.staging(g, &sfs);
        launch_yuv420_to_bgr(stage, yuv_planes_of(S), sfs, (int)n, g.rows, g.cols, dst, g.pitch, g.frame_bytes, q);
    } else {
        launch_yuv420_to_bgr(src, yuv_planes_of(*f.yuv), f.stride, (int)n, g.rows, g.cols, dst, g.pitch, g.frame_bytes, q);
    }
    return cudaGetLastError();
}

cudaError_t frames_in(const Geometry& g, const FrameFmt& f, const uint8_t* src, long n, uint8_t* dst, uint8_t* stage, cudaStream_t q) {
    const cudaError_t e = frames_in_transfer(g, f, src, n, dst, stage, q);
    return e != cudaSuccess ? e : frames_in_convert(g, f, src, n, dst, stage, q);
}

// output, convert: BGR frames at `src` -> YUV, into `stage` (host) or into the caller's frames at `dst` (device)
cudaError_t frames_out_convert(const Geometry& g, const FrameFmt& f, const uint8_t* src, long n, uint8_t* dst, uint8_t* stage,
                               cudaStream_t q) {
    if (!f.yuv) return cudaSuccess;
    if (f.host) {
        size_t sfs = 0;
        const vstab_yuv_layout S = f.staging(g, &sfs);
        launch_bgr_to_yuv420(src, g.pitch, g.frame_bytes, (int)n, g.rows, g.cols, stage, yuv_planes_of(S), sfs, q);
    } else {
        launch_bgr_to_yuv420(src, g.pitch, g.frame_bytes, (int)n, g.rows, g.cols, dst, yuv_planes_of(*f.yuv), f.stride, q);
    }
    return cudaGetLastError();
}

// output, transfer: -> the caller's frames at `dst`, from the BGR frames at `src` (BGR) or from `stage` (host YUV)
cudaError_t frames_out_transfer(const Geometry& g, const FrameFmt& f, const uint8_t* src, long n, uint8_t* dst, const uint8_t* stage,
                                cudaStream_t q) {
    if (!f.yuv)
        return bgr_copy(dst, f.step, f.stride, src, g.pitch, g.frame_bytes, n, g.rows, g.cols,
                        f.host ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice, q);
    if (!f.host) return cudaSuccess;
    size_t sfs = 0;
    const vstab_yuv_layout S = f.staging(g, &sfs);
    return yuv_copy(dst, *f.yuv, f.stride, stage, S, sfs, n, g.rows, g.cols, cudaMemcpyDeviceToHost, q);
}

cudaError_t frames_out(const Geometry& g, const FrameFmt& f, const uint8_t* src, long n, uint8_t* dst, uint8_t* stage, cudaStream_t q) {
    const cudaError_t e = frames_out_convert(g, f, src, n, dst, stage, q);
    return e != cudaSuccess ? e : frames_out_transfer(g, f, src, n, dst, stage, q);
}

// ---- ORB / SIFT registration (stabilizer.cpp:440-787), shared by the streaming instance and the offline runner ---------
// The reference set is one packed device buffer: {int count, pad to 16 B} {OrbKeypoint[kOrbMaxKp]} {u8 desc[kOrbMaxKp][128]},
// so the offline ranks can broadcast it as it is.
constexpr size_t kRefPackKps = 16;
constexpr size_t kRefPackDesc = kRefPackKps + sizeof(OrbKeypoint) * kOrbMaxKp;
constexpr size_t kRefPackBytes = kRefPackDesc + (size_t)128 * kOrbMaxKp;
struct RefSet {
    int* count;
    OrbKeypoint* kps;
    uint8_t* desc;
    explicit RefSet(void* pack)
        : count((int*)pack), kps((OrbKeypoint*)((char*)pack + kRefPackKps)), desc((uint8_t*)pack + kRefPackDesc) {}
};

// Everything one registration in flight needs.  The front ends are replayed as CUDA graphs keyed on their buffers and
// stream (run_graphed), so a lane passes the same buffers from call to call.
struct RegLane {
    OrbPlan* orb = nullptr;              // plan of the mode, created on its first use
    SiftPlan* sift = nullptr;
    DevBuf feat_ws, feat_gray, kps, desc, counts, m_idx, m_d0, m_d1, m_good, m_ref, m_cur, m_status, fit;
    cudaStream_t q = nullptr;            // own stream (offline lanes beyond the first), or null: the caller's
    cudaEvent_t done = nullptr;
    ~RegLane() {
        if (q) { cudaStreamSynchronize(q); cudaStreamDestroy(q); }
        if (done) cudaEventDestroy(done);
        if (orb) orb_plan_destroy(orb);
        if (sift) sift_plan_destroy(sift);
    }
    int* ncur() { return counts.as<int>(); }
    int* nmatch() { return counts.as<int>() + 1; }
    double* Tfit() { return fit.as<double>(); }
    int* fitc() { return reinterpret_cast<int*>(fit.as<double>() + 16); }
    uint8_t* gray(const Geometry& g, int slot) { return feat_gray.as<uint8_t>() + (size_t)slot * g.ww * g.wh; }

    // buffers (on first use: `gray_slots` conditioned images, counts zeroed on `stream`) and the plan of `mode`
    vstab_status setup(Geometry& g, int mode, int gray_slots, cudaStream_t stream, std::string& err) {
        auto set_err = [&](const std::string& e) { err = e; };
        if (!feat_ws.p) {
            CK(g.nn_tables());
            CK(feat_ws.alloc(featprep_workspace_bytes(g.ww, g.wh)));
            CK(feat_gray.alloc((size_t)g.ww * g.wh * gray_slots));
            CK(kps.alloc(sizeof(OrbKeypoint) * kOrbMaxKp));
            CK(desc.alloc(128 * kOrbMaxKp));                                    // 32 B (ORB) or 128 B (SIFT) per row
            CK(counts.alloc(sizeof(int) * 2));                                  // {ncur, nmatch}
            CK(m_idx.alloc(4 * kOrbMaxKp)); CK(m_d0.alloc(4 * kOrbMaxKp)); CK(m_d1.alloc(l2_match_scratch_bytes(kOrbMaxKp, 1)));   // m_d1: second distances (Hamming) / matcher scratch (L2)
            CK(m_good.alloc(kOrbMaxKp)); CK(m_status.alloc(kOrbMaxKp));
            CK(m_ref.alloc(sizeof(float2) * kOrbMaxKp)); CK(m_cur.alloc(sizeof(float2) * kOrbMaxKp));
            CK(fit.alloc(sizeof(double) * 16 + sizeof(int) * 4));              // T[9], M[6], counts[2]
            CK(cudaMemsetAsync(counts.p, 0, sizeof(int) * 2, stream));
        }
        if (mode == VSTAB_ORB_FULL_LOCK && !orb && !(orb = orb_plan_create(g.ww, g.wh, 0.10, kOrbMaxKp, &err)))    // MAX_KEYPOINT_RELATIVE_SIZE_ORB, :493
            return VSTAB_ERR_CUDA;
        if (mode == VSTAB_SIFT_FULL_LOCK && !sift && !(sift = sift_plan_create(g.ww, g.wh, 0.05, kOrbMaxKp, &err)))  // MAX_KEYPOINT_RELATIVE_SIZE_SIFT, :507
            return VSTAB_ERR_CUDA;
        return VSTAB_OK;
    }

    // condition `frame` (:448-477) into gray slot `slot` and detect + describe it into kps / desc / *count
    void detect(Geometry& g, const uint8_t* frame, size_t step, int slot, bool is_orb, OrbKeypoint* k, uint8_t* d, int* count,
                bool reference_order, cudaStream_t st) {
        launch_featprep(frame, step, g.nn_x.as<int>(), g.nn_y.as<int>(), g.ww, g.wh, feat_ws.p, gray(g, slot), st);
        if (is_orb) launch_orb(orb, gray(g, slot), k, d, count, reference_order, st);               // :557-559 / :604-612
        else launch_sift(sift, gray(g, slot), k, d, count, st);                                      // :572-574 / :614-621
    }

    // reference capture (:520-589): the ORB set in cv::ORB's order
    void capture(Geometry& g, const uint8_t* frame, size_t step, int slot, bool is_orb, const RefSet& ref, cudaStream_t st) {
        detect(g, frame, step, slot, is_orb, ref.kps, ref.desc, ref.count, true, st);
    }

    // detect + describe, match against `ref` (:647-716) and fit (:734-758) into Tfit / fitc.  False, having launched no
    // matcher, when the SIFT matcher could not be launched (kL2MapErr).
    bool match(Geometry& g, const uint8_t* frame, size_t step, int slot, bool is_orb, const RefSet& ref, cudaStream_t st) {
        detect(g, frame, step, slot, is_orb, kps.as<OrbKeypoint>(), desc.as<uint8_t>(), ncur(), false, st);
        if (is_orb)
            launch_hamming_match(ref.desc, ref.count, ref.kps, desc.as<uint8_t>(), ncur(), kps.as<OrbKeypoint>(), kOrbMaxKp, 0.6f,
                                 m_idx.as<int>(), m_d0.as<int>(), m_d1.as<int>(), m_good.as<uint8_t>(), m_ref.as<float2>(),
                                 m_cur.as<float2>(), m_status.as<uint8_t>(), nmatch(), st);
        else if (!launch_l2_match(ref.desc, ref.count, ref.kps, desc.as<uint8_t>(), ncur(), kps.as<OrbKeypoint>(), kOrbMaxKp, m_d1.p,
                                  m_idx.as<int>(), m_d0.as<int>(), m_good.as<uint8_t>(), m_ref.as<float2>(), m_cur.as<float2>(),
                                  m_status.as<uint8_t>(), nmatch(), st))
            return false;
        launch_fit_large(m_ref.as<float2>(), m_cur.as<float2>(), m_status.as<uint8_t>(), nmatch(), 5.0, g.ww / 2.0, g.wh / 2.0,
                         Tfit(), Tfit() + 9, fitc(), st);
        return true;
    }
};

}  // namespace

// =====================================================================================
// streaming instance
// =====================================================================================
struct vstab {
    int device = 0;
    cudaStream_t stream = nullptr;       // estimation stream: ingest -> pyramid -> LK -> fit -> corner detection
    cudaStream_t out_stream = nullptr;   // output stream: smoothing / lock -> warp -> device-to-host copy
    cudaEvent_t ev_in = nullptr;         // input frame is in the ring (caller may reuse its buffer)
    cudaEvent_t ev_fit[8] = {};          // [n & 7]: T[n] and the channel sums of frame n are final
    cudaEvent_t ev_out = nullptr;        // output chain of the previous call has finished reading the ring
    cudaStream_t gftt_stream[2] = {};    // corner detection of frame n on [n & 1]: beside LK / fit and beside frame n+1's
    cudaStream_t copy_stream = nullptr;  // upload of frame n, beside everything else
    cudaStream_t ing_stream = nullptr;   // ingest -> pyramid of frame n, beside the tracker of frame n-1 and the next upload
    // ORB / SIFT registration one call ahead: the presentation frame of call n+1 is already in the ring during call n
    // (future >= 1), so its registration is enqueued on feat_stream right after the smoothing of call n and overlaps the
    // download of call n, the host's return and the next upload.  lock_h / lock_tap are double-buffered by call parity.
    cudaStream_t feat_stream = nullptr;
    cudaEvent_t ev_feat = nullptr;       // look-ahead registration finished
    cudaEvent_t ev_reg = nullptr;        // this call's registration / smoothing no longer needs the scratch buffers
    long feat_p = -1;                    // presentation frame the pending look-ahead result belongs to
    bool feat_pending = false;           // something was enqueued on feat_stream since the last wait
    int lock_slot = 0;                   // lock_h / lock_tap half of the current call
    // Output prepared one call ahead (host-buffer calls, LK-path modes, future >= 1): everything the output of call n+1
    // reads is already on the device when call n has enqueued its estimation, so its smoothing / lock + warp run on
    // pre_stream beside the download of call n and call n+1 only has to copy out.  wp / dout are double-buffered;
    // setStabilizationMode / setTrail bump `epoch` and the prepared frame is dropped (the output is then built inside
    // the call as before).
    cudaStream_t pre_stream = nullptr;
    cudaEvent_t ev_pre = nullptr;        // prepared output (and its ACCUMULATED product update) is complete
    cudaEvent_t ev_chain = nullptr;      // in-call output chain has left the lock / smoothing state behind
    bool pre_valid = false;
    long pre_call = -1;
    unsigned long pre_epoch = 0, epoch = 0;
    long pre_acc_to = -1;                // accumulatedTransform_.to_frame_idx once the prepared output is presented
    int out_slot = 0;                    // half of wp / dout that holds the latest presented output
    cudaEvent_t ev_pyr[4] = {};          // [n & 3]: gray pyramid (and channel sums) of frame n are complete
    cudaEvent_t ev_gftt[4] = {};         // [n & 3]: corners of frame n are complete (needed by LK of frame n+1)
    size_t P = 15, F = 15;
    int working_height = 360;
    int mode = VSTAB_GLOBAL_SMOOTHING;
    long lock_call = 0;          // call index at which the current mode was set
    bool acc_valid = false;      // accumulatedTransform_.H non-empty
    long acc_to = -1;            // accumulatedTransform_.to_frame_idx
    long acc_call = -1;          // call whose update of the accumulated product has been enqueued
    long n = 0;                  // number of frames pushed so far == index of the next call
    long last_presented = 0;
    bool inited = false;
    Geometry g;
    long W = 0;                  // window size in frames
    DevBuf ring, sums, pyrs[3], corners0, corners1, ccount, lkpts, lkstat, T, Mtap, fitc, acc, wp, gmem[2], dout, dout1;
    WarpParams* wp_at(int slot) { return wp.as<WarpParams>() + (slot & 1); }
    uint8_t* dout_at(int slot) { return (slot & 1) ? dout1.as<uint8_t>() : dout.as<uint8_t>(); }
    long t_mod = 0;
    GfttWorkspace gws[2] = {};   // [n & 1]: the corner detections of two consecutive frames overlap
    // ORB / SIFT registration state (reference: referenceGray_/Keypoints_/Descriptors_, hpp:447-456, and the
    // function-static previouslyReturnedH, cpp:446 -- per instance here).  One lane serves the in-call (out_stream) and the
    // look-ahead (feat_stream) registration, ordered by ev_reg / ev_feat; its conditioned image is double-buffered by
    // lock_slot like lock_h / lock_tap.
    RegLane reg;
    DevBuf ref, lock_h, lock_tap;        // ref: packed reference set (RefSet)
    bool has_reference = false;
    bool trail = false;                     // copyFeathered branch of stabilizeFrame (:1303-1307)
    bool partial_fix = false;               // TRANSLATION_/ROTATION_LOCK fed with the accumulated lock (hpp:23 @todo)
    DevBuf trail_bg, trail_ws;              // trail_background_ (:129) and K14 scratch
    // auto-crop (vstab_set_crop): on when crop.max_zoom > 1.  crop_need holds n_j of call j in slot j % (R + 1); crop_reset:
    // the next output chain first sets the whole history to 1 (calls before the enabling call need no zoom)
    CropArgs crop{1.0, 0.0, 0};
    bool crop_reset = false;
    DevBuf crop_need;
    // staging of host YUV frames (FrameFmt): the input frame is uploaded here (copy_stream) and converted into the ring, the
    // presented BGR frame is converted here (out_stream) and downloaded.  One frame each: every use is ordered by its stream.
    DevBuf yuv_in, yuv_out;
    std::string err;
    // VSTAB_TRACE=1: host wall-clock split of the streaming call (printed by vstab_destroy)
    double trace_us[4] = {0, 0, 0, 0};   // enqueue output chain | enqueue upload + estimation | wait upload | wait output
    long trace_calls = 0;
    // device-side marks of one call (timing events): 0 upload start, 1 upload end, 2 estimation start, 3 pyramid done,
    // 4 LK+fit done, 5 corners start, 6 corners done, 7 output start, 8 smoothing done, 9 warp done, 10 download done
    // (two sets, alternating per call: the marks of call n-1 are read at the end of call n, without draining the pipeline)
    cudaEvent_t tev[2][13] = {};
    double tev_ms[13] = {};              // [10]: upload start of the next call (the period); [11] LK start, [12] LK done
    long tev_calls = 0;
    void mark(int i, cudaStream_t q) {
        if (!tev[0][0]) return;
        cudaEventRecord(tev[n & 1][i], q);
    }

    void set_err(const std::string& e) { err = e; }
    uint8_t* pyr(long frame) { return pyrs[frame % 3].as<uint8_t>(); }   // three: frame n+1's is built while LK reads n-1, n
    float2* corners(int i) { return (i & 1) ? corners1.as<float2>() : corners0.as<float2>(); }
};

static vstab_status stream_init(vstab* s, int rows, int cols) {
    auto set_err = [&](const std::string& e) { s->err = e; };
    vstab_status st = s->g.init(rows, cols, s->working_height, s->err);
    if (st != VSTAB_OK) return st;
    Geometry& g = s->g;
    s->W = (long)(s->P + 1 + s->F);
    s->t_mod = s->W + 2;
    CK(s->ring.alloc(g.frame_bytes * (size_t)s->W + 64));
    CK(s->sums.alloc(sizeof(unsigned long long) * 3 * s->W));
    for (auto& b : s->pyrs) CK(b.alloc(g.pd.frame_bytes));
    CK(s->corners0.alloc(sizeof(float2) * kMaxCorners));
    CK(s->corners1.alloc(sizeof(float2) * kMaxCorners));
    CK(s->ccount.alloc(sizeof(int) * 2));
    CK(s->lkpts.alloc(sizeof(float2) * kMaxCorners));
    CK(s->lkstat.alloc(kMaxCorners));
    CK(s->T.alloc(sizeof(double) * 9 * s->t_mod));
    CK(s->Mtap.alloc(sizeof(double) * 6));
    CK(s->fitc.alloc(sizeof(int) * 2));
    CK(s->acc.alloc(sizeof(double) * 9));
    CK(s->wp.alloc(sizeof(WarpParams) * 2));
    CK(s->dout.alloc(g.frame_bytes + 64));
    CK(s->dout1.alloc(g.frame_bytes + 64));
    for (int i = 0; i < 2; ++i) {
        size_t gbytes = gftt_workspace_bytes(g.ww, g.wh, g.min_distance, 1, &s->gws[i]);
        CK(s->gmem[i].alloc(gbytes));
        gftt_bind_workspace(s->gmem[i].p, &s->gws[i]);
    }
    CK(cudaMemsetAsync(s->ccount.p, 0, sizeof(int) * 2, s->stream));
    CK(cudaMemsetAsync(s->T.p, 0, sizeof(double) * 9 * s->t_mod, s->stream));
    CK(cudaStreamSynchronize(s->stream));          // the chains of the first call start on other streams
    s->inited = true;
    return VSTAB_OK;
}

// A streaming call is a set of chains with no loop-carried dependency between frames except LK(n) <- corners(n-1)
// (SURVEY Appendix C: with future >= 1 the output of call n depends only on transforms up to n-1, because the
// reference's window average excludes the newest transform, stabilizer.cpp:825-826, and ACCUMULATED lock uses T[n-F]):
//   copy_stream:        upload of frame n
//   ing_stream:         [upload n] -> ingest -> pyramid                                 (three pyramid buffers)
//   s->stream:          [pyramid n, corners n-1] -> LK against frame n-1 -> fit T[n]
//   gftt_stream[n & 1]: [pyramid n] -> corner detection of frame n                      (two workspaces: frames overlap)
//   out_stream / pre_stream: lock / window average -> warp of frame n-F -> copy out
// so the host only waits for the upload and the copy-out, and the per-frame latency of the one-CTA corner selection
// (~140 us) or of the tracker is not the call rate.  With future == 0 the output chain waits for T[n] of this call.

// Estimation of frame index s->n whose pixels are in ring slot n % W once s->ev_in has fired.
static vstab_status stream_estimate(vstab* s) {
    auto set_err = [&](const std::string& e) { s->err = e; };
    Geometry& g = s->g;
    cudaStream_t q = s->stream;
    const long n = s->n;
    const long slot = n % s->W;
    const int cur = (int)(n & 1), prev = cur ^ 1;
    const uint8_t* frame = s->ring.as<uint8_t>() + (size_t)slot * g.frame_bytes;
    unsigned long long* sums = s->sums.as<unsigned long long>() + slot * 3;
    int* ccount = s->ccount.as<int>();
    cudaStream_t up = s->ing_stream;
    CK(cudaStreamWaitEvent(up, s->ev_in, 0));
    // pyramid buffer n % 3 held frame n-3: read by LK of frames n-3 and n-2 and by the corner detection of n-3
    if (n >= 3) {
        CK(cudaStreamWaitEvent(up, s->ev_fit[(n - 2) & 7], 0));
        CK(cudaStreamWaitEvent(up, s->ev_gftt[(n - 3) & 3], 0));
    }
    s->mark(2, up);
    CK(cudaMemsetAsync(sums, 0, sizeof(unsigned long long) * 3, up));
    launch_ingest(g.plan, frame, g.pitch, g.frame_bytes, 1, s->pyr(n), g.pd.frame_bytes, sums, up);    // :1169-1175
    launch_pyramid(g.pd, s->pyr(n), 1, up);
    CK(cudaEventRecord(s->ev_pyr[n & 3], up));
    s->mark(3, up);
    CK(cudaStreamWaitEvent(q, s->ev_pyr[n & 3], 0));
    if (n > 0) {
        CK(cudaStreamWaitEvent(q, s->ev_gftt[(n - 1) & 3], 0));       // corners of frame n-1
        s->mark(11, q);
        // :1187 trackFeatures
        launch_lk(s->pyr(n - 1), s->pyr(n), g.pd.frame_bytes, g.pd.frame_bytes, g.pd, s->corners(prev), ccount + prev, 1,
                  s->lkpts.as<float2>(), s->lkstat.as<uint8_t>(), q);
        s->mark(12, q);
        // :1203 estimateMotion, :1209 updateTransformations
        launch_fit(s->corners(prev), s->lkpts.as<float2>(), s->lkstat.as<uint8_t>(), ccount + prev, 1, 3.0,
                   g.ww / 2.0, g.wh / 2.0, s->T.as<double>() + (size_t)(n % s->t_mod) * 9, s->Mtap.as<double>(),
                   s->fitc.as<int>(), nullptr, n, q);
    }
    CK(cudaEventRecord(s->ev_fit[n & 7], q));
    s->mark(4, q);
    // corner detection of this frame (:1318 / :1179) only feeds the next call's tracker.  Its corner list (parity n & 1)
    // was last read by the tracker / fit of frame n-1.
    cudaStream_t qg = s->gftt_stream[cur];
    CK(cudaStreamWaitEvent(qg, s->ev_pyr[n & 3], 0));
    if (n > 0) CK(cudaStreamWaitEvent(qg, s->ev_fit[(n - 1) & 7], 0));
    s->mark(5, qg);
    static const bool tap_eig = getenv("VSTAB_DEBUG_TAPS") != nullptr;   // the min-eigenvalue map is a debug tap only
    launch_gftt(s->pyr(n), g.pd.frame_bytes, g.ww, g.wh, 1, 0.01, g.min_distance, kMaxCorners, s->gws[cur],
                s->corners(cur), ccount + cur, tap_eig ? s->gws[cur].eig : nullptr, qg);
    CK(cudaEventRecord(s->ev_gftt[n & 3], qg));
    s->mark(6, qg);
    CK(cudaGetLastError());
    return VSTAB_OK;
}

// calculateFullLockStabilization, ORB / SIFT branch (stabilizer.cpp:440-787) for presentation frame p, on
// the output stream: condition the full-resolution frame, detect + describe, and either capture the
// reference (first call after setStabilizationMode) or match against it and fit.
static vstab_status stream_feature_lock(vstab* s, long p, cudaStream_t q, int slot) {
    auto set_err = [&](const std::string& e) { s->err = e; };
    Geometry& g = s->g;
    RegLane& L = s->reg;
    const bool is_orb = s->mode == VSTAB_ORB_FULL_LOCK;
    if (!s->ref.p) {
        CK(s->ref.alloc(kRefPackBytes));
        CK(s->lock_h.alloc(sizeof(double) * 9 * 2));
        CK(s->lock_tap.alloc(sizeof(int) * 8 * 2));
        CK(cudaMemsetAsync(s->ref.p, 0, kRefPackBytes, q));
    }
    vstab_status st = L.setup(g, s->mode, 2, q, s->err);
    if (st != VSTAB_OK) return st;
    const uint8_t* frame = s->ring.as<uint8_t>() + (size_t)(p % s->W) * g.frame_bytes;           // :444
    const RefSet ref(s->ref.p);
    double* lock_h = s->lock_h.as<double>() + 9 * slot;
    int* lock_tap = s->lock_tap.as<int>() + 8 * slot;
    if (!s->has_reference) {                                                                     // :520-589
        L.capture(g, frame, g.pitch, slot, is_orb, ref, q);
        launch_lock_update(L.Tfit(), L.fitc(), ref.count, ref.count, ref.count, 1, lock_h, lock_tap, q);
        s->has_reference = true;
    } else {
        // "previously returned H" (:446) carries over from the other half
        CK(cudaMemcpyAsync(lock_h, s->lock_h.as<double>() + 9 * (slot ^ 1), sizeof(double) * 9, cudaMemcpyDeviceToDevice, q));
        if (!L.match(g, frame, g.pitch, slot, is_orb, ref, q)) { s->err = kL2MapErr; return VSTAB_ERR_CUDA; }
        launch_lock_update(L.Tfit(), L.fitc(), ref.count, L.ncur(), L.nmatch(), 0, lock_h, lock_tap, q);  // :784-787
    }
    CK(cudaGetLastError());
    return VSTAB_OK;
}

// Output chain of call s->n (n >= 1) on s->out_stream; `d_out`/`out_pitch`: where the warped
// presentation frame goes.  The caller has already made out_stream wait for the transforms it needs.
// Output chain of call n on stream q: lock / window average -> warp of the presentation frame into d_out, its warp
// parameters into *wp.  `ahead`: enqueued during call n-1 (no trace marks, `last_presented` moves when it is consumed).
static vstab_status stream_output(vstab* s, long n, uint8_t* d_out, size_t out_pitch, WarpParams* wp, cudaStream_t q,
                                  bool prepared_ahead) {
    auto set_err = [&](const std::string& e) { s->err = e; };
    Geometry& g = s->g;
    const long p = n - (long)s->F > 0 ? n - (long)s->F : 0;                                            // :1226-1229
    if (!prepared_ahead) s->mark(7, q);
    const bool partial = s->partial_fix && (s->mode == VSTAB_TRANSLATION_LOCK || s->mode == VSTAB_ROTATION_LOCK);
    if (s->mode == VSTAB_ACCUMULATED_FULL_LOCK || partial) {                                           // :317-338
        // (acc_call == n: a prepared-ahead chain that was dropped afterwards has already made this call's update)
        if (s->acc_call != n) launch_acc_update(s->T.as<double>(), s->t_mod, p, s->acc_valid ? 0 : 1, s->acc.as<double>(), q);
        s->acc_call = n;
        if (prepared_ahead) {
            s->pre_acc_to = p;                 // host-side view moves when the prepared output is consumed
        } else {
            s->acc_valid = true;
            s->acc_to = p;
        }
    }
    const bool feature_lock = s->mode == VSTAB_ORB_FULL_LOCK || s->mode == VSTAB_SIFT_FULL_LOCK;
    if (feature_lock) {
        const int slot = s->lock_slot ^ 1;
        const bool ahead = s->feat_pending && s->feat_p == p && s->has_reference;
        if (s->feat_pending) CK(cudaStreamWaitEvent(q, s->ev_feat, 0));     // look-ahead result, or just the scratch buffers
        s->feat_pending = false;
        if (!ahead) {
            vstab_status st = stream_feature_lock(s, p, q, slot);
            if (st != VSTAB_OK) return st;
        }
        s->lock_slot = slot;
    }
    SmoothArgs a{};
    a.T = s->T.as<double>(); a.t_mod = s->t_mod;
    a.P = (int)s->P; a.F = (int)s->F;
    a.mode = s->mode; a.lock_call = s->lock_call;
    a.acc = s->acc.as<double>(); a.acc_mod = 0;
    a.lock_h = feature_lock ? s->lock_h.as<double>() + 9 * s->lock_slot : nullptr;
    a.scale = g.scale;
    a.sums = s->sums.as<unsigned long long>(); a.sums_mod = s->W; a.frame_base = 0;
    a.npix = (double)g.rows * (double)g.cols;
    a.partial_fix = s->partial_fix ? 1 : 0;
    a.cx = (double)(float)(g.ww / 2.0); a.cy = (double)(float)(g.wh / 2.0);                            // Point2f centre
    launch_smooth(a, n, 1, wp, q);                                                                     // :1234-1296
    if (s->crop.max_zoom > 1.0) {
        // one history slot per call, written by the chain that builds the call: a prepared output that is dropped and
        // rebuilt writes the same slot again, and successive chains are ordered by ev_pre / ev_chain
        if (!s->crop_need.p) CK(s->crop_need.alloc(sizeof(double) * (kCropMaxR + 1)));
        CropArgs ca = s->crop;
        ca.rows = g.rows; ca.cols = g.cols;
        ca.need = s->crop_need.as<double>(); ca.need_base = 0; ca.need_mod = ca.R + 1;
        ca.reset = s->crop_reset ? 1 : 0;
        s->crop_reset = false;
        launch_crop(ca, nullptr, 0, wp, n, 1, q);
    }
    if (!prepared_ahead) s->mark(8, q);
    if (feature_lock && s->F >= 2 && s->has_reference) {
        // registration of the next call's presentation frame, beside this call's warp and download.  Only with
        // future >= 2: that frame (n + 1 - F <= n - 1) is then already in the ring; with future == 1 it is the frame
        // this very call uploads AFTER its output chain was enqueued, so its registration stays inside call n + 1
        const long pn = n + 1 - (long)s->F > 0 ? n + 1 - (long)s->F : 0;
        CK(cudaEventRecord(s->ev_reg, q));
        CK(cudaStreamWaitEvent(s->feat_stream, s->ev_reg, 0));
        vstab_status st = stream_feature_lock(s, pn, s->feat_stream, s->lock_slot ^ 1);
        if (st != VSTAB_OK) return st;
        CK(cudaEventRecord(s->ev_feat, s->feat_stream));
        s->feat_p = pn;
        s->feat_pending = true;
    }
    if (s->trail) {
        // presentation_output = copyFeathered(presentation_image, trail_background_, H); trail_background_ = its clone (:1303-1307)
        if (!s->trail_bg.p) {
            CK(s->trail_bg.alloc(g.frame_bytes + 64));
            CK(s->trail_ws.alloc(trail_workspace_bytes(g.cols, g.rows, g.frame_bytes)));
            CK(cudaMemsetAsync(s->trail_bg.p, 0, g.frame_bytes, q));                                   // Mat::zeros, :128-130
        }
        launch_trail(s->ring.as<uint8_t>(), g.pitch, g.frame_bytes, s->W, wp, -1, s->trail_bg.as<uint8_t>(),
                     g.cols, g.rows, s->trail_ws.p, d_out, out_pitch, q);
        CK(cudaMemcpy2DAsync(s->trail_bg.p, g.pitch, d_out, out_pitch, (size_t)g.cols * 3, g.rows, cudaMemcpyDeviceToDevice, q));
    } else {
        launch_warp(s->ring.as<uint8_t>(), g.pitch, g.frame_bytes, s->W, wp, 1, g.cols, g.rows,
                    d_out, out_pitch, 0, q);                                                           // :1309-1313
    }
    if (!prepared_ahead) s->mark(9, q);
    CK(cudaGetLastError());
    if (!prepared_ahead) s->last_presented = p;
    return VSTAB_OK;
}

// One stabilizeFrame call: frame `in` in the caller's format `in_fmt`, its output into `out` in `out_fmt`.  A call on host
// frames returns when `out` is complete.
static vstab_status stream_call(vstab* s, const uint8_t* in, const FrameFmt& in_fmt, uint8_t* out, const FrameFmt& out_fmt) {
    auto set_err = [&](const std::string& e) { s->err = e; };
    Geometry& g = s->g;
    uint8_t* slot = s->ring.as<uint8_t>() + (size_t)(s->n % s->W) * g.frame_bytes;
    const bool host_wait = in_fmt.host;
    const bool direct_out = out_fmt.direct();          // the warp writes the caller's BGR buffer itself
    const bool out_first = s->n > 0 && s->F >= 1;      // output chain does not need this call's transform
    if (!s->yuv_in.p && in_fmt.staging_bytes(g)) CK(s->yuv_in.alloc(in_fmt.staging_bytes(g)));
    if (!s->yuv_out.p && out_fmt.staging_bytes(g)) CK(s->yuv_out.alloc(out_fmt.staging_bytes(g)));
    static const bool trace = getenv("VSTAB_TRACE") != nullptr;
    auto now_us = [] { return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    const double tr0 = trace ? now_us() : 0.0;
    double tr1 = 0.0;
    if (trace && !s->tev[0][0])
        for (auto& set : s->tev) for (auto& e : set) cudaEventCreate(&e);
    // which fit the output chain of call c has to wait for.  The window average reads T up to c-1
    // (stabilizer.cpp:825-826); every other mode reads nothing newer than the presentation frame p = c - F (its T for
    // the ACCUMULATED product, its channel sums, its pixels).  Waiting for the fit of frame c-1 or c-2 there would tie
    // the call period to the LATENCY of a frame's estimation (upload -> pyramid -> LK -> fit, ~0.4 ms, longer than two
    // calls); with a lag of min(F, 6) frames only its throughput matters.
    auto fit_event = [&](long c) {
        long lag = (long)s->F < 6 ? (long)s->F : 6;
        // ORB / SIFT lock also registers the NEXT call's presentation frame c + 1 - F from the ring (look-ahead)
        if (s->mode == VSTAB_ORB_FULL_LOCK || s->mode == VSTAB_SIFT_FULL_LOCK) lag -= 1;
        if (s->mode == VSTAB_GLOBAL_SMOOTHING || lag < 1) lag = 1;
        if (lag > c) lag = c;
        return s->ev_fit[(c - lag) & 7];
    };
    auto output_into = [&](long c, int slot, cudaStream_t q, bool ahead) -> vstab_status {
        uint8_t* dst = direct_out ? out : s->dout_at(slot);
        return stream_output(s, c, dst, direct_out ? out_fmt.step : g.pitch, s->wp_at(slot), q, ahead);
    };
    // the presented BGR half -> `out` on out_stream, unless the warp wrote it there (an output prepared one call ahead
    // did not know the caller's format)
    auto copy_out = [&](int slot) -> vstab_status {
        if (!direct_out) CK(frames_out(g, out_fmt, s->dout_at(slot), 1, out, s->yuv_out.as<uint8_t>(), s->out_stream));
        return VSTAB_OK;
    };

    if (s->pre_valid) CK(cudaStreamWaitEvent(s->out_stream, s->ev_pre, 0));   // used or not, its state updates come first
    bool in_call_chain = false;                                               // ev_chain: that chain's lock state is final
    if (out_first) {
        const long p = s->n - (long)s->F > 0 ? s->n - (long)s->F : 0;
        if (s->pre_valid && s->pre_call == s->n && s->pre_epoch == s->epoch && !direct_out) {
            s->out_slot ^= 1;                                          // prepared during the previous call
            s->last_presented = p;
            if (s->mode == VSTAB_ACCUMULATED_FULL_LOCK || (s->partial_fix && (s->mode == VSTAB_TRANSLATION_LOCK || s->mode == VSTAB_ROTATION_LOCK))) {
                s->acc_valid = true; s->acc_to = s->pre_acc_to;
            }
            s->mark(7, s->out_stream); s->mark(8, s->out_stream); s->mark(9, s->out_stream);
        } else {
            CK(cudaStreamWaitEvent(s->out_stream, fit_event(s->n), 0));
            s->out_slot ^= 1;
            vstab_status st = output_into(s->n, s->out_slot, s->out_stream, false);
            if (st != VSTAB_OK) return st;
            CK(cudaEventRecord(s->ev_chain, s->out_stream));
            in_call_chain = true;
        }
        vstab_status st = copy_out(s->out_slot);
        if (st != VSTAB_OK) return st;
    }
    s->pre_valid = false;
    if (trace) tr1 = now_us();
    // estimation chain.  The ring slot being overwritten held frame n-W; its readers (the warp and the
    // channel sums of an earlier call's output chain) are ordered before this copy by ev_out.
    // Host input: the upload runs on its own stream, beside the estimation of the previous frame.
    // (Enqueuing the upload ahead of the output chain was measured: no gain for LK, -4 % for ORB lock.)
    cudaStream_t up = s->copy_stream;
    if (s->n > 0) CK(cudaStreamWaitEvent(up, s->ev_out, 0));
    s->mark(0, up);
    CK(frames_in(g, in_fmt, in, 1, slot, s->yuv_in.as<uint8_t>(), up));
    s->mark(1, up);
    CK(cudaEventRecord(s->ev_in, up));
    vstab_status st = stream_estimate(s);
    if (st != VSTAB_OK) return st;
    if (!out_first) {
        if (s->n == 0) {
            // call 0 returns the input frame itself (:1181)
            CK(cudaStreamWaitEvent(s->out_stream, s->ev_in, 0));
            CK(frames_out(g, out_fmt, slot, 1, out, s->yuv_out.as<uint8_t>(), s->out_stream));
            s->last_presented = 0;
        } else {
            CK(cudaStreamWaitEvent(s->out_stream, s->ev_fit[s->n & 7], 0));   // future == 0: needs T[n] of this call
            s->out_slot ^= 1;
            st = output_into(s->n, s->out_slot, s->out_stream, false);
            if (st != VSTAB_OK) return st;
            CK(cudaEventRecord(s->ev_chain, s->out_stream));
            in_call_chain = true;
            st = copy_out(s->out_slot);
            if (st != VSTAB_OK) return st;
        }
    }
    // the next call's output, beside this call's download (see pre_stream)
    const bool lk_mode = s->mode != VSTAB_ORB_FULL_LOCK && s->mode != VSTAB_SIFT_FULL_LOCK;
    if (host_wait && out_fmt.host && s->F >= 1 && lk_mode && !s->trail) {
        const long c = s->n + 1;
        if (in_call_chain) CK(cudaStreamWaitEvent(s->pre_stream, s->ev_chain, 0));
        CK(cudaStreamWaitEvent(s->pre_stream, fit_event(c), 0));
        st = output_into(c, s->out_slot ^ 1, s->pre_stream, true);
        if (st != VSTAB_OK) return st;
        CK(cudaEventRecord(s->ev_pre, s->pre_stream));
        s->pre_valid = true; s->pre_call = c; s->pre_epoch = s->epoch;
    }
    s->mark(10, s->out_stream);
    CK(cudaEventRecord(s->ev_out, s->out_stream));
    const double tr2 = trace ? now_us() : 0.0;
    if (host_wait) {
        CK(cudaEventSynchronize(s->ev_in));                            // caller may reuse `in` (the reference clones, :160)
        const double tr3 = trace ? now_us() : 0.0;
        CK(cudaStreamSynchronize(s->out_stream));                      // `out` is complete
        if (trace) {
            const double tr4 = now_us();
            s->trace_us[0] += tr1 - tr0; s->trace_us[1] += tr2 - tr1; s->trace_us[2] += tr3 - tr2; s->trace_us[3] += tr4 - tr3;
            s->trace_calls += 1;
            // device-side marks of the previous call relative to its upload start (skipped while its corner
            // detection is still running)
            const int pv = (int)((s->n - 1) & 1), cu = (int)(s->n & 1);
            if (out_first && s->n > 3 && cudaEventQuery(s->tev[pv][6]) == cudaSuccess && cudaEventQuery(s->tev[pv][4]) == cudaSuccess) {
                for (int i = 1; i <= 10; ++i) {
                    float ms = 0.f;
                    if (cudaEventElapsedTime(&ms, s->tev[pv][0], s->tev[pv][i]) == cudaSuccess) s->tev_ms[i - 1] += ms;
                }
                float ms = 0.f;
                if (cudaEventElapsedTime(&ms, s->tev[pv][0], s->tev[cu][0]) == cudaSuccess) s->tev_ms[10] += ms;
                if (cudaEventElapsedTime(&ms, s->tev[pv][0], s->tev[pv][11]) == cudaSuccess) s->tev_ms[11] += ms;
                if (cudaEventElapsedTime(&ms, s->tev[pv][0], s->tev[pv][12]) == cudaSuccess) s->tev_ms[12] += ms;
                s->tev_calls += 1;
            }
        }
    }
    s->n += 1;
    return VSTAB_OK;
}

// The vstab_stabilize_frame* entry points: argument checks, device, set-up on the first call, then the call
static vstab_status stream_entry(vstab* s, const uint8_t* in, const FrameFmt& in_fmt, int rows, int cols, uint8_t* out,
                                 const FrameFmt& out_fmt) {
    if (!s) return VSTAB_ERR_INVALID_ARGUMENT;
    if (!in || !out) { s->err = "null image pointer"; return VSTAB_ERR_INVALID_ARGUMENT; }
    if (rows <= 10 || cols <= 10) {                                                                    // :99-103
        s->err = "Stabilizer: Frame has invalid size. Rows: " + std::to_string(rows) + ", Cols: " + std::to_string(cols);
        return VSTAB_ERR_INVALID_ARGUMENT;
    }
    vstab_status st = in_fmt.check(rows, cols, false, s->err);
    if (st == VSTAB_OK) st = out_fmt.check(rows, cols, false, s->err);
    if (st != VSTAB_OK) return st;
    if (s->inited && (s->g.rows != rows || s->g.cols != cols)) {                                        // :110-112
        s->err = "Stabilizer: Frame size has changed. This is not supported.";
        return VSTAB_ERR_SIZE_CHANGED;
    }
    const bool acc_mode = s->mode == VSTAB_ACCUMULATED_FULL_LOCK ||
                          (s->partial_fix && (s->mode == VSTAB_TRANSLATION_LOCK || s->mode == VSTAB_ROTATION_LOCK));
    if (acc_mode && s->acc_valid) {
        // the reference asserts presentation_frame_idx > 0 and from_frame_idx == acc.to (:329-332);
        // both fail exactly when the presentation frame did not advance (SURVEY B.6)
        const long p = s->n - (long)s->F > 0 ? s->n - (long)s->F : 0;
        if (p != s->acc_to + 1) {
            s->err = "ACCUMULATED_FULL_LOCK before the window can advance (reference asserts, stabilizer.cpp:329)";
            return VSTAB_ERR_STATE;
        }
    }
    auto set_err = [&](const std::string& e) { s->err = e; };
    CK(cudaSetDevice(s->device));
    if (!s->inited && (st = stream_init(s, rows, cols)) != VSTAB_OK) return st;
    return stream_call(s, in, in_fmt, out, out_fmt);
}

extern "C" {

int vstab_abi_version(void) { return VSTAB_ABI_VERSION; }

const char* vstab_status_string(vstab_status st) {
    switch (st) {
        case VSTAB_OK: return "ok";
        case VSTAB_ERR_INVALID_ARGUMENT: return "invalid argument";
        case VSTAB_ERR_SIZE_CHANGED: return "frame size changed";
        case VSTAB_ERR_CUDA: return "CUDA error";
        case VSTAB_ERR_UNSUPPORTED: return "unsupported";
        case VSTAB_ERR_NCCL: return "NCCL error";
        case VSTAB_ERR_STATE: return "invalid state";
    }
    return "?";
}

vstab_status vstab_create(size_t past_frames, size_t future_frames, int working_height, int device, vstab_t** out) {
    if (!out) return VSTAB_ERR_INVALID_ARGUMENT;
    *out = nullptr;
    // argument checks of Stabilizer::Stabilizer, stabilizer.cpp:40-49
    if (past_frames == 0 && future_frames == 0) { g_err = "Stabilizer: pastFrames and futureFrames cannot both be 0"; return VSTAB_ERR_INVALID_ARGUMENT; }
    if ((double)working_height <= 90.0) { g_err = "Stabilizer: workingHeight must be greater than 90.000000"; return VSTAB_ERR_INVALID_ARGUMENT; }
    if (working_height > 2160) { g_err = "Stabilizer: workingHeight must be no more than 2160"; return VSTAB_ERR_INVALID_ARGUMENT; }
    if (!device_ok(device, g_err)) return VSTAB_ERR_CUDA;
    vstab* s = new (std::nothrow) vstab();
    if (!s) return VSTAB_ERR_CUDA;
    s->device = device; s->P = past_frames; s->F = future_frames; s->working_height = working_height;
    // the tracker / fit chain and the output chain are on the critical path of a call; corner detection has a whole
    // call of slack, so it runs at the lowest priority and yields SMs to them
    int prio_least = 0, prio_greatest = 0;
    cudaDeviceGetStreamPriorityRange(&prio_least, &prio_greatest);
    if (cudaStreamCreateWithPriority(&s->stream, cudaStreamNonBlocking, prio_greatest) != cudaSuccess ||
        cudaStreamCreateWithPriority(&s->out_stream, cudaStreamNonBlocking, prio_greatest) != cudaSuccess ||
        cudaEventCreateWithFlags(&s->ev_in, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s->ev_fit[0], cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s->ev_fit[1], cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s->ev_fit[2], cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s->ev_fit[3], cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s->ev_fit[4], cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s->ev_fit[5], cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s->ev_fit[6], cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s->ev_fit[7], cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s->ev_out, cudaEventDisableTiming) != cudaSuccess ||
        cudaStreamCreateWithPriority(&s->gftt_stream[0], cudaStreamNonBlocking, prio_least) != cudaSuccess ||
        cudaStreamCreateWithPriority(&s->gftt_stream[1], cudaStreamNonBlocking, prio_least) != cudaSuccess ||
        cudaStreamCreateWithFlags(&s->copy_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithPriority(&s->ing_stream, cudaStreamNonBlocking, prio_greatest) != cudaSuccess ||
        cudaStreamCreateWithPriority(&s->feat_stream, cudaStreamNonBlocking, prio_greatest) != cudaSuccess ||
        cudaEventCreateWithFlags(&s->ev_feat, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s->ev_reg, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s->ev_pyr[0], cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s->ev_pyr[1], cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s->ev_pyr[2], cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s->ev_pyr[3], cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s->ev_gftt[1], cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s->ev_gftt[2], cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s->ev_gftt[3], cudaEventDisableTiming) != cudaSuccess ||
        cudaStreamCreateWithPriority(&s->pre_stream, cudaStreamNonBlocking, prio_greatest) != cudaSuccess ||
        cudaEventCreateWithFlags(&s->ev_pre, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s->ev_chain, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s->ev_gftt[0], cudaEventDisableTiming) != cudaSuccess) {
        g_err = "cudaStreamCreate failed"; vstab_destroy(s); return VSTAB_ERR_CUDA;
    }
    *out = s;
    return VSTAB_OK;
}

void vstab_destroy(vstab_t* s) {
    if (!s) return;
    cudaSetDevice(s->device);
    if (s->trace_calls > 0)
        fprintf(stderr, "[vstab trace] %ld calls, per call: enqueue-output %.1f us, enqueue-upload+estimation %.1f us, "
                        "wait-upload %.1f us, wait-output %.1f us\n", s->trace_calls, s->trace_us[0] / s->trace_calls,
                s->trace_us[1] / s->trace_calls, s->trace_us[2] / s->trace_calls, s->trace_us[3] / s->trace_calls);
    if (s->tev_calls > 0) {
        static const char* nm[10] = {"upload end", "estimation start", "pyramid done", "LK+fit done", "corners start",
                                     "corners done", "output start", "smoothing done", "warp done", "download done"};
        fprintf(stderr, "[vstab trace] device marks of a call relative to its upload start (us, %ld calls):", s->tev_calls);
        for (int i = 0; i < 10; ++i) fprintf(stderr, " %s %.1f;", nm[i], 1e3 * s->tev_ms[i] / s->tev_calls);
        fprintf(stderr, " LK start %.1f; LK done %.1f; next upload start %.1f\n", 1e3 * s->tev_ms[11] / s->tev_calls,
                1e3 * s->tev_ms[12] / s->tev_calls, 1e3 * s->tev_ms[10] / s->tev_calls);
    }
    if (s->stream) { cudaStreamSynchronize(s->stream); cudaStreamDestroy(s->stream); }
    if (s->out_stream) { cudaStreamSynchronize(s->out_stream); cudaStreamDestroy(s->out_stream); }
    if (s->ev_in) cudaEventDestroy(s->ev_in);
    for (auto e : s->ev_fit) if (e) cudaEventDestroy(e);
    if (s->ev_out) cudaEventDestroy(s->ev_out);
    for (auto q : s->gftt_stream) if (q) { cudaStreamSynchronize(q); cudaStreamDestroy(q); }
    if (s->copy_stream) { cudaStreamSynchronize(s->copy_stream); cudaStreamDestroy(s->copy_stream); }
    if (s->ing_stream) { cudaStreamSynchronize(s->ing_stream); cudaStreamDestroy(s->ing_stream); }
    if (s->feat_stream) { cudaStreamSynchronize(s->feat_stream); cudaStreamDestroy(s->feat_stream); }
    if (s->ev_feat) cudaEventDestroy(s->ev_feat);
    if (s->ev_reg) cudaEventDestroy(s->ev_reg);
    for (auto e : s->ev_pyr) if (e) cudaEventDestroy(e);
    for (auto e : s->ev_gftt) if (e) cudaEventDestroy(e);
    if (s->pre_stream) { cudaStreamSynchronize(s->pre_stream); cudaStreamDestroy(s->pre_stream); }
    if (s->ev_pre) cudaEventDestroy(s->ev_pre);
    if (s->ev_chain) cudaEventDestroy(s->ev_chain);
    for (auto& set : s->tev) for (auto& e : set) if (e) cudaEventDestroy(e);     // VSTAB_TRACE marks
    delete s;
}

vstab_status vstab_set_mode(vstab_t* s, int mode) {
    if (!s) return VSTAB_ERR_INVALID_ARGUMENT;
    if (mode < 0 || mode > 5) { s->err = "Stabilizer: Invalid stabilization mode"; return VSTAB_ERR_INVALID_ARGUMENT; }
    // stabilizer.cpp:55-70: reset reference + accumulator, keep window / prevGray_ / prevPoints_
    s->has_reference = false;
    s->feat_p = -1;                      // a pending look-ahead registration belongs to the old reference: not consumed
    s->acc_valid = false;
    s->acc_to = -1;
    s->acc_call = -1;
    s->epoch += 1;                       // an output prepared ahead under the old mode is dropped
    s->mode = mode;
    s->lock_call = s->n;
    return VSTAB_OK;
}

int vstab_get_mode(const vstab_t* s) { return s ? s->mode : -1; }

size_t vstab_total_frame_window_size(const vstab_t* s) { return s ? s->P + 1 + s->F : 0; }

vstab_status vstab_synchronize(vstab_t* s) {
    if (!s) return VSTAB_ERR_INVALID_ARGUMENT;
    auto set_err = [&](const std::string& e) { s->err = e; };
    CK(cudaSetDevice(s->device));
    CK(cudaStreamSynchronize(s->stream));
    CK(cudaStreamSynchronize(s->out_stream));
    CK(cudaStreamSynchronize(s->gftt_stream[0]));
    CK(cudaStreamSynchronize(s->gftt_stream[1]));
    CK(cudaStreamSynchronize(s->copy_stream));
    CK(cudaStreamSynchronize(s->ing_stream));
    CK(cudaStreamSynchronize(s->feat_stream));
    CK(cudaStreamSynchronize(s->pre_stream));
    return VSTAB_OK;
}

vstab_status vstab_stabilize_frame(vstab_t* s, const uint8_t* bgr, int rows, int cols, size_t step,
                                   uint8_t* out_bgr, size_t out_step) {
    return stream_entry(s, bgr, {true, nullptr, step}, rows, cols, out_bgr, {true, nullptr, out_step});
}

vstab_status vstab_stabilize_frame_device(vstab_t* s, const uint8_t* d_bgr, int rows, int cols, size_t step,
                                          uint8_t* d_out_bgr, size_t out_step) {
    return stream_entry(s, d_bgr, {false, nullptr, step}, rows, cols, d_out_bgr, {false, nullptr, out_step});
}

size_t vstab_yuv_layout_packed(int format, int rows, int cols, vstab_yuv_layout* out) {
    std::string err;
    vstab_yuv_layout L;
    if (!out || rows <= 0 || cols <= 0 || (format != VSTAB_PIX_NV12 && format != VSTAB_PIX_I420)) return 0;
    const size_t bytes = yuv_packed(format, rows, cols, &L);
    if (!yuv_extent(&L, rows, cols, err)) return 0;             // odd sizes
    *out = L;
    return bytes;
}

vstab_status vstab_stabilize_frame_yuv(vstab_t* s, const uint8_t* in, const vstab_yuv_layout* in_layout, int rows, int cols,
                                       uint8_t* out, const vstab_yuv_layout* out_layout) {
    if (s && (!in_layout || !out_layout)) { s->err = "null YUV layout"; return VSTAB_ERR_INVALID_ARGUMENT; }   // FrameFmt: BGR
    return stream_entry(s, in, {true, in_layout}, rows, cols, out, {true, out_layout});
}

vstab_status vstab_stabilize_frame_yuv_device(vstab_t* s, const uint8_t* d_in, const vstab_yuv_layout* in_layout, int rows,
                                              int cols, uint8_t* d_out, const vstab_yuv_layout* out_layout) {
    if (s && (!in_layout || !out_layout)) { s->err = "null YUV layout"; return VSTAB_ERR_INVALID_ARGUMENT; }
    return stream_entry(s, d_in, {false, in_layout}, rows, cols, d_out, {false, out_layout});
}

int vstab_decompose_homography(const double H[9], double cx, double cy, vstab_hparams* out) {
    if (!H || !out) return -1;
    HParams hp;
    if (!decompose_h(H, cx, cy, &hp)) return 0;
    out->s = hp.s; out->theta = hp.theta; out->k = hp.k; out->delta = hp.delta;
    out->t[0] = hp.t[0]; out->t[1] = hp.t[1]; out->v[0] = hp.v[0]; out->v[1] = hp.v[1];
    return 1;
}

void vstab_compose_homography(const vstab_hparams* p, double cx, double cy, double H[9]) {
    if (!p || !H) return;
    HParams hp;
    hp.s = p->s; hp.theta = p->theta; hp.k = p->k; hp.delta = p->delta;
    hp.t[0] = p->t[0]; hp.t[1] = p->t[1]; hp.v[0] = p->v[0]; hp.v[1] = p->v[1];
    compose_h(&hp, cx, cy, H);
}

const char* vstab_last_error(const vstab_t* s) { return s ? s->err.c_str() : g_err.c_str(); }

void* vstab_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) return nullptr;
    return p;
}
void vstab_host_free(void* p) { if (p) cudaFreeHost(p); }

int vstab_working_width(const vstab_t* s) { return s && s->inited ? s->g.ww : 0; }
int vstab_working_height(const vstab_t* s) { return s && s->inited ? s->g.wh : 0; }
long vstab_presentation_index(const vstab_t* s) { return s ? s->last_presented : -1; }

long vstab_read_tap(vstab_t* s, int tap, void* dst, size_t dst_bytes) {
    if (!s || !s->inited || !dst || s->n == 0) return -1;
    if (cudaSetDevice(s->device) != cudaSuccess) return -1;
    if (cudaStreamSynchronize(s->stream) != cudaSuccess) return -1;
    if (cudaStreamSynchronize(s->out_stream) != cudaSuccess) return -1;
    if (cudaStreamSynchronize(s->gftt_stream[0]) != cudaSuccess || cudaStreamSynchronize(s->gftt_stream[1]) != cudaSuccess) return -1;
    if (cudaStreamSynchronize(s->copy_stream) != cudaSuccess || cudaStreamSynchronize(s->ing_stream) != cudaSuccess) return -1;
    Geometry& g = s->g;
    const long last = s->n - 1;                 // index of the most recent frame
    const int cur = (int)(last & 1), prev = cur ^ 1;
    auto copy = [&](const void* src, size_t bytes, long count) -> long {
        if (bytes > dst_bytes) return -2;
        if (cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
        return count;
    };
    int counts[2] = {0, 0};
    if (cudaMemcpy(counts, s->ccount.p, sizeof(counts), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
    switch (tap) {
        case VSTAB_TAP_GRAY: return copy(s->pyr(last) + g.pd.off[0], (size_t)g.ww * g.wh, (long)g.ww * g.wh);
        case VSTAB_TAP_PYR1: case VSTAB_TAP_PYR2: case VSTAB_TAP_PYR3: {
            const int l = tap - VSTAB_TAP_PYR1 + 1;
            return copy(s->pyr(last) + g.pd.off[l], (size_t)g.pd.w[l] * g.pd.h[l], (long)g.pd.w[l] * g.pd.h[l]);
        }
        case VSTAB_TAP_PREV_PTS: if (last == 0) return 0; return copy(s->corners(prev), sizeof(float2) * counts[prev], counts[prev]);
        case VSTAB_TAP_LK_PTS: if (last == 0) return 0; return copy(s->lkpts.p, sizeof(float2) * counts[prev], counts[prev]);
        case VSTAB_TAP_LK_STATUS: if (last == 0) return 0; return copy(s->lkstat.p, counts[prev], counts[prev]);
        case VSTAB_TAP_NEW_PTS: return copy(s->corners(cur), sizeof(float2) * counts[cur], counts[cur]);
        case VSTAB_TAP_T: if (last == 0) return 0; return copy(s->T.as<double>() + (size_t)(last % s->t_mod) * 9, sizeof(double) * 9, 9);
        case VSTAB_TAP_M: if (last == 0) return 0; return copy(s->Mtap.p, sizeof(double) * 6, 6);
        case VSTAB_TAP_H_STABILIZE: if (last == 0) return 0; return copy((char*)s->wp_at(s->out_slot) + offsetof(WarpParams, Hw), sizeof(double) * 9, 9);
        case VSTAB_TAP_H_SCALED: if (last == 0) return 0; return copy((char*)s->wp_at(s->out_slot) + offsetof(WarpParams, Hs), sizeof(double) * 9, 9);
        case VSTAB_TAP_BORDER: if (last == 0) return 0; return copy((char*)s->wp_at(s->out_slot) + offsetof(WarpParams, border), 3, 3);
        case VSTAB_TAP_EIG: return copy(s->gws[cur].eig, sizeof(float) * g.ww * g.wh, (long)g.ww * g.wh);
        case VSTAB_TAP_INLIERS: if (last == 0) return 0; return copy(s->fitc.p, sizeof(int) * 2, 2);
        case VSTAB_TAP_LOCK_H: if (!s->lock_h.p) return 0; return copy(s->lock_h.as<double>() + 9 * s->lock_slot, sizeof(double) * 9, 9);
        case VSTAB_TAP_ORB_COUNTS: if (!s->lock_tap.p) return 0; return copy(s->lock_tap.as<int>() + 8 * s->lock_slot, sizeof(int) * 5, 5);
        case VSTAB_TAP_FEAT_GRAY: if (!s->reg.feat_gray.p) return 0; return copy(s->reg.gray(g, s->lock_slot), (size_t)g.ww * g.wh, (long)g.ww * g.wh);
        case VSTAB_TAP_CHANNEL_SUMS:
            return copy(s->sums.as<unsigned long long>() + (s->last_presented % s->W) * 3, sizeof(unsigned long long) * 3, 3);
    }
    return -1;
}

}  // extern "C"

// =====================================================================================
// offline (frame-sharded) runner
// =====================================================================================
struct vstab_offline {
    int device = 0;
    cudaStream_t stream = nullptr;
    size_t P = 0, F = 0;
    int max_batch = 0;
    Geometry g;
    DevBuf pyr, corners, ccount, lkpts, lkstat, Mtap, fitc, wp, gmem, acc, halo_sums;
    GfttWorkspace gws{};
    long acc_n_total = 0, acc_anchor = -1;
    size_t acc_capacity = 0;
    const double* acc_T = nullptr;
    int last_ncalls = 0;
    StageTimer timer;
    // ORB / SIFT registration (offline): packed reference set (RefSet) and its mode, gathered registrations
    int ref_mode = -1;
    DevBuf ref_pack;
    const double* reg_all = nullptr;
    long reg_n = 0;
    // registration lanes: frames of a shard are independent units, so vstab_offline_register deals them round-robin to
    // lanes; lane 0 runs on `stream` (it also captures the reference set), every other one on a stream of its own
    std::vector<std::unique_ptr<RegLane>> lanes;
    cudaEvent_t ev_reg_fork = nullptr;
    // sharded job (vstab_offline_run, vstab_offline_run_host): NCCL communicator of this rank, chunk ring, output chunks and
    // YUV staging kept between runs; the streams of the fused pass (source: copy_in, warp: copy_out) and of downloads to a
    // host sink
    void* comm = nullptr;
    int rank = 0, world = 1;
    DevBuf job_chunk, job_out, job_stage;
    size_t job_chunk_frames = 0, job_out_frames = 0, job_stage_bytes = 0;
    cudaStream_t copy_in = nullptr, copy_out = nullptr, download = nullptr;
    // YUV layouts of the frames of run_host / run (vstab_offline_set_yuv; none: BGR)
    std::optional<vstab_yuv_layout> yin, yout;
    // auto-crop (vstab_offline_set_crop): every render recomputes the warp parameters of the R calls before its first one
    // (crop_halo) and their needs (crop_need, halo + batch), so no state is carried from one render to the next
    CropArgs crop{1.0, 0.0, 0};
    DevBuf crop_halo, crop_need;
    std::string err;
    void set_err(const std::string& e) { err = e; }
};

// the first K registration lanes, set up for `mode`
static vstab_status offline_lanes(vstab_offline* o, int mode, int K) {
    auto set_err = [&](const std::string& e) { o->err = e; };
    while ((int)o->lanes.size() < K) {
        std::unique_ptr<RegLane> L(new (std::nothrow) RegLane());
        if (!L) { o->err = "out of memory"; return VSTAB_ERR_CUDA; }
        if (!o->lanes.empty()) {
            CK(cudaStreamCreateWithFlags(&L->q, cudaStreamNonBlocking));
            CK(cudaEventCreateWithFlags(&L->done, cudaEventDisableTiming));
        }
        o->lanes.push_back(std::move(L));
    }
    for (int k = 0; k < K; ++k) {
        RegLane& L = *o->lanes[k];
        vstab_status st = L.setup(o->g, mode, 1, L.q ? L.q : o->stream, o->err);
        if (st != VSTAB_OK) return st;
    }
    return VSTAB_OK;
}

// the reference set and lane 0 (which captures it) for `mode`
static vstab_status offline_feature_setup(vstab_offline* o, int mode) {
    auto set_err = [&](const std::string& e) { o->err = e; };
    if (mode != VSTAB_ORB_FULL_LOCK && mode != VSTAB_SIFT_FULL_LOCK) { o->err = "mode must be ORB_FULL_LOCK or SIFT_FULL_LOCK"; return VSTAB_ERR_INVALID_ARGUMENT; }
    if (!o->ref_pack.p) {
        CK(o->ref_pack.alloc(kRefPackBytes));
        CK(cudaMemsetAsync(o->ref_pack.p, 0, kRefPackBytes, o->stream));
    }
    return offline_lanes(o, mode, 1);
}

extern "C" {

size_t vstab_offline_reference_bytes(void) { return kRefPackBytes; }

// Reference capture (stabilizer.cpp:520-589) from the anchor frame (the presentation frame of the call at
// which the mode was set); the owner of that frame calls this, exports the packed set, and the other
// ranks import it after the broadcast.
vstab_status vstab_offline_reference_capture(vstab_offline_t* o, const uint8_t* d_frame, size_t step, int mode) {
    if (!o || !d_frame) return VSTAB_ERR_INVALID_ARGUMENT;
    auto set_err = [&](const std::string& e) { o->err = e; };
    CK(cudaSetDevice(o->device));
    vstab_status st = offline_feature_setup(o, mode);
    if (st != VSTAB_OK) return st;
    o->lanes[0]->capture(o->g, d_frame, step, 0, mode == VSTAB_ORB_FULL_LOCK, RefSet(o->ref_pack.p), o->stream);
    CK(cudaGetLastError());
    o->ref_mode = mode;
    return VSTAB_OK;
}

vstab_status vstab_offline_reference_export(vstab_offline_t* o, void* d_pack) {
    if (!o || !d_pack || !o->ref_pack.p) return VSTAB_ERR_INVALID_ARGUMENT;
    auto set_err = [&](const std::string& e) { o->err = e; };
    CK(cudaSetDevice(o->device));
    CK(cudaMemcpyAsync(d_pack, o->ref_pack.p, kRefPackBytes, cudaMemcpyDeviceToDevice, o->stream));
    return VSTAB_OK;
}

vstab_status vstab_offline_reference_import(vstab_offline_t* o, const void* d_pack, int mode) {
    if (!o || !d_pack) return VSTAB_ERR_INVALID_ARGUMENT;
    auto set_err = [&](const std::string& e) { o->err = e; };
    CK(cudaSetDevice(o->device));
    vstab_status st = offline_feature_setup(o, mode);
    if (st != VSTAB_OK) return st;
    CK(cudaMemcpyAsync(o->ref_pack.p, d_pack, kRefPackBytes, cudaMemcpyDeviceToDevice, o->stream));
    o->ref_mode = mode;
    return VSTAB_OK;
}

// Register frames d_frames[0..n) against the reference set (stabilizer.cpp:604-787 without the carry):
// d_reg[i] = {inverse(H with scale forced to 1) [9], valid} -- identity / 0 when the reference would have
// returned its previous matrix.
vstab_status vstab_offline_register(vstab_offline_t* o, const uint8_t* d_frames, size_t frame_stride, size_t step, int n,
                                    double* d_reg) {
    if (!o || !d_frames || !d_reg || n < 1) return VSTAB_ERR_INVALID_ARGUMENT;
    auto set_err = [&](const std::string& e) { o->err = e; };
    if (o->ref_mode != VSTAB_ORB_FULL_LOCK && o->ref_mode != VSTAB_SIFT_FULL_LOCK) { o->err = "no reference set: call vstab_offline_reference_capture / _import first"; return VSTAB_ERR_STATE; }
    CK(cudaSetDevice(o->device));
    cudaStream_t q = o->stream;
    const RefSet ref(o->ref_pack.p);
    const bool is_orb = o->ref_mode == VSTAB_ORB_FULL_LOCK;
    // lanes: the ORB front end is ~44 small dependent launches per frame, SIFT at 4K mostly large ones (and 1.1 GB of pyramid per
    // lane).  Measured on B200, complete offline pass, frames/s with 1 / 2 / 3 / 4 / 8 lanes: ORB 1080p 1950 / - / 2834 / 2981 / 3117,
    // SIFT 4K 442 / 511 / 531 / - / 563.
    int K = is_orb ? 8 : 4;
    if (K > n) K = n;
    vstab_status st = offline_lanes(o, o->ref_mode, K);
    if (st != VSTAB_OK) return st;
    if (K > 1) {
        if (!o->ev_reg_fork) CK(cudaEventCreateWithFlags(&o->ev_reg_fork, cudaEventDisableTiming));
        CK(cudaEventRecord(o->ev_reg_fork, q));                       // reference set, frames: ordered before every lane
        for (int k = 1; k < K; ++k) CK(cudaStreamWaitEvent(o->lanes[k]->q, o->ev_reg_fork, 0));
    }
    for (int i = 0; i < n; ++i) {
        RegLane& L = *o->lanes[i % K];
        cudaStream_t ql = L.q ? L.q : q;
        if (!L.match(o->g, d_frames + (size_t)i * frame_stride, step, 0, is_orb, ref, ql)) { o->err = kL2MapErr; return VSTAB_ERR_CUDA; }
        launch_reg_store(L.Tfit(), L.fitc(), ref.count, L.ncur(), L.nmatch(), d_reg + (size_t)i * 10, ql);
    }
    for (int k = 1; k < K; ++k) {
        CK(cudaEventRecord(o->lanes[k]->done, o->lanes[k]->q));
        CK(cudaStreamWaitEvent(q, o->lanes[k]->done, 0));
    }
    CK(cudaGetLastError());
    return VSTAB_OK;
}

// All registrations of the clip ({H[9], valid} per frame, e.g. after the all-gather) for vstab_offline_render
// in ORB_FULL_LOCK / SIFT_FULL_LOCK.
vstab_status vstab_offline_set_registrations(vstab_offline_t* o, const double* d_reg_all, long n_total) {
    if (!o) return VSTAB_ERR_INVALID_ARGUMENT;
    o->reg_all = d_reg_all; o->reg_n = n_total;
    return VSTAB_OK;
}

vstab_status vstab_offline_create(size_t past_frames, size_t future_frames, int working_height, int rows, int cols,
                                  int max_batch, int device, vstab_offline_t** out) {
    if (!out) return VSTAB_ERR_INVALID_ARGUMENT;
    *out = nullptr;
    if (past_frames == 0 && future_frames == 0) { g_err = "Stabilizer: pastFrames and futureFrames cannot both be 0"; return VSTAB_ERR_INVALID_ARGUMENT; }
    if ((double)working_height <= 90.0 || working_height > 2160) { g_err = "Stabilizer: workingHeight out of range"; return VSTAB_ERR_INVALID_ARGUMENT; }
    if (rows <= 10 || cols <= 10 || max_batch < 1) { g_err = "invalid frame size or batch"; return VSTAB_ERR_INVALID_ARGUMENT; }
    if (!device_ok(device, g_err)) return VSTAB_ERR_CUDA;
    vstab_offline* o = new (std::nothrow) vstab_offline();
    if (!o) return VSTAB_ERR_CUDA;
    auto fail = [&](vstab_status st, const std::string& m) { g_err = m; vstab_offline_destroy(o); return st; };
    o->device = device; o->P = past_frames; o->F = future_frames; o->max_batch = max_batch;
    if (cudaStreamCreateWithFlags(&o->stream, cudaStreamNonBlocking) != cudaSuccess) return fail(VSTAB_ERR_CUDA, "cudaStreamCreate failed");
    vstab_status st = o->g.init(rows, cols, working_height, g_err);
    if (st != VSTAB_OK) { vstab_offline_destroy(o); return st; }
    Geometry& g = o->g;
    const size_t nb = (size_t)max_batch + 1;   // + halo
    bool ok = o->pyr.alloc(g.pd.frame_bytes * nb) == cudaSuccess &&
              o->corners.alloc(sizeof(float2) * kMaxCorners * nb) == cudaSuccess &&
              o->ccount.alloc(sizeof(int) * nb) == cudaSuccess &&
              o->lkpts.alloc(sizeof(float2) * kMaxCorners * nb) == cudaSuccess &&
              o->lkstat.alloc(kMaxCorners * nb) == cudaSuccess &&
              o->Mtap.alloc(sizeof(double) * 6 * nb) == cudaSuccess &&
              o->fitc.alloc(sizeof(int) * 2 * nb) == cudaSuccess &&
              o->wp.alloc(sizeof(WarpParams) * nb) == cudaSuccess &&
              o->halo_sums.alloc(sizeof(unsigned long long) * 3) == cudaSuccess;
    if (!ok) return fail(VSTAB_ERR_CUDA, "cudaMalloc(offline buffers) failed");
    size_t gbytes = gftt_workspace_bytes(g.ww, g.wh, g.min_distance, (int)nb, &o->gws);
    if (o->gmem.alloc(gbytes) != cudaSuccess) return fail(VSTAB_ERR_CUDA, "cudaMalloc(gftt workspace) failed");
    gftt_bind_workspace(o->gmem.p, &o->gws);
    *out = o;
    return VSTAB_OK;
}

void vstab_offline_destroy(vstab_offline_t* o) {
    if (!o) return;
    cudaSetDevice(o->device);
    if (o->stream) { cudaStreamSynchronize(o->stream); cudaStreamDestroy(o->stream); }
    if (o->copy_in) { cudaStreamSynchronize(o->copy_in); cudaStreamDestroy(o->copy_in); }
    if (o->copy_out) { cudaStreamSynchronize(o->copy_out); cudaStreamDestroy(o->copy_out); }
    if (o->download) { cudaStreamSynchronize(o->download); cudaStreamDestroy(o->download); }
    if (o->ev_reg_fork) cudaEventDestroy(o->ev_reg_fork);
    if (o->comm) nccl_comm_destroy(o->comm);
    delete o;
}

uintptr_t vstab_offline_stream(vstab_offline_t* o) { return o ? (uintptr_t)o->stream : 0; }

vstab_status vstab_offline_synchronize(vstab_offline_t* o) {
    if (!o) return VSTAB_ERR_INVALID_ARGUMENT;
    auto set_err = [&](const std::string& e) { o->err = e; };
    CK(cudaSetDevice(o->device));
    CK(cudaStreamSynchronize(o->stream));
    return VSTAB_OK;
}

}  // extern "C"

// d_sums: [n][3] u64 per-channel byte sums of the n frames (device), may be NULL
extern "C" vstab_status vstab_offline_estimate(vstab_offline_t* o, const uint8_t* d_frames, size_t frame_stride,
                                                size_t step, int n, long first, const uint8_t* d_halo,
                                                double* d_T, unsigned long long* d_sums) {
    if (!o || !d_frames || !d_T || n < 1) return VSTAB_ERR_INVALID_ARGUMENT;
    auto set_err = [&](const std::string& e) { o->err = e; };
    if (n > o->max_batch) { o->err = "n exceeds max_batch"; return VSTAB_ERR_INVALID_ARGUMENT; }
    if (first > 0 && !d_halo) { o->err = "halo frame required when first > 0"; return VSTAB_ERR_INVALID_ARGUMENT; }
    if (step < (size_t)o->g.cols * 3) { o->err = "row step smaller than 3*cols"; return VSTAB_ERR_INVALID_ARGUMENT; }
    CK(cudaSetDevice(o->device));
    Geometry& g = o->g;
    cudaStream_t q = o->stream;
    uint8_t* pyr = o->pyr.as<uint8_t>();
    // pyramid slot 0 = halo (frame first-1), slots 1..n = the batch
    const bool has_halo = first > 0;
    if (d_sums) CK(cudaMemsetAsync(d_sums, 0, sizeof(unsigned long long) * 3 * n, q));
    unsigned long long* sums = d_sums;
    if (!sums) {
        // sums are a by-product of the ingest pass; without a destination use scratch in wp
        sums = (unsigned long long*)o->wp.p;
        CK(cudaMemsetAsync(sums, 0, sizeof(unsigned long long) * 3 * n, q));
    }
    if (has_halo) {
        CK(cudaMemsetAsync(o->halo_sums.p, 0, sizeof(unsigned long long) * 3, q));
        launch_ingest(g.plan, d_halo, step, 0, 1, pyr, g.pd.frame_bytes, o->halo_sums.as<unsigned long long>(), q);
    }
    o->timer.begin(ST_INGEST, q);
    launch_ingest(g.plan, d_frames, step, frame_stride, n, pyr + g.pd.frame_bytes, g.pd.frame_bytes, sums, q);
    o->timer.end(ST_INGEST, q);
    const int s0 = has_halo ? 0 : 1;              // first pyramid slot in use
    const int nslots = has_halo ? n + 1 : n;
    // corners of every "previous" frame of a pair: slots s0 .. n-1
    const int npairs = nslots - 1;
    float2* corners = o->corners.as<float2>() + (size_t)s0 * kMaxCorners;
    int* ccount = o->ccount.as<int>() + s0;
    o->timer.begin(ST_PYRAMID, q);
    launch_pyramid(g.pd, pyr + (size_t)s0 * g.pd.frame_bytes, nslots, q);
    o->timer.end(ST_PYRAMID, q);
    if (npairs > 0) {
        o->timer.begin(ST_GFTT, q);
        launch_gftt(pyr + (size_t)s0 * g.pd.frame_bytes, g.pd.frame_bytes, g.ww, g.wh, npairs, 0.01, g.min_distance,
                    kMaxCorners, o->gws, corners, ccount, nullptr, q);
        o->timer.end(ST_GFTT, q);
        o->timer.begin(ST_LK, q);
        launch_lk(pyr + (size_t)s0 * g.pd.frame_bytes, pyr + (size_t)(s0 + 1) * g.pd.frame_bytes, g.pd.frame_bytes,
                  g.pd.frame_bytes, g.pd, corners, ccount, npairs, o->lkpts.as<float2>(), o->lkstat.as<uint8_t>(), q);
        o->timer.end(ST_LK, q);
        // pair i (slots s0+i, s0+i+1) -> T of frame first + (s0 + i + 1 - 1) = first + s0 + i
        o->timer.begin(ST_FIT, q);
        launch_fit(corners, o->lkpts.as<float2>(), o->lkstat.as<uint8_t>(), ccount, npairs, 3.0, g.ww / 2.0, g.wh / 2.0,
                   d_T + (size_t)s0 * 9, o->Mtap.as<double>(), o->fitc.as<int>(), nullptr, first + s0, q);
        o->timer.end(ST_FIT, q);
    }
    if (!has_halo) {
        // T[0] = identity (never used: SURVEY Appendix C)
        static const double I9[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
        CK(cudaMemcpyAsync(d_T, I9, sizeof(I9), cudaMemcpyHostToDevice, q));
    }
    CK(cudaGetLastError());
    return VSTAB_OK;
}

// d_sums: [.][3] u64 indexed like d_frames (frame - frame_base)
static vstab_status offline_render_impl(vstab_offline_t* o, const uint8_t* d_frames, size_t frame_stride,
                                        size_t step, long frame_base, int n, long call_first,
                                        const double* d_T_all, long n_total, int mode, long lock_call,
                                        const unsigned long long* d_sums,
                                        uint8_t* d_out, size_t out_frame_stride, size_t out_step,
                                        unsigned long long* d_check /* [n] pre-zeroed, or null */,
                                        long slot_mod = 0 /* > 0: d_frames is a ring, frame f sits in slot (f - frame_base) % slot_mod */,
                                        cudaStream_t on = nullptr /* stream of the two launches; null: the instance stream */) {
    if (!o || !d_frames || !d_T_all || !d_out || !d_sums || n < 1) return VSTAB_ERR_INVALID_ARGUMENT;
    auto set_err = [&](const std::string& e) { o->err = e; };
    if (n > o->max_batch + 1) { o->err = "n exceeds max_batch"; return VSTAB_ERR_INVALID_ARGUMENT; }
    if (mode < 0 || mode > 5) { o->err = "Stabilizer: Invalid stabilization mode"; return VSTAB_ERR_INVALID_ARGUMENT; }
    const bool feature_lock = mode == VSTAB_ORB_FULL_LOCK || mode == VSTAB_SIFT_FULL_LOCK;
    if (feature_lock && (!o->reg_all || o->reg_n != n_total)) {
        o->err = "call vstab_offline_set_registrations(d_reg_all, n_total) before rendering in ORB / SIFT lock";
        return VSTAB_ERR_STATE;
    }
    if (mode == VSTAB_ACCUMULATED_FULL_LOCK && lock_call < (long)o->F) {
        o->err = "ACCUMULATED_FULL_LOCK must be set at a call index >= future (SURVEY B.6)"; return VSTAB_ERR_STATE;
    }
    CK(cudaSetDevice(o->device));
    Geometry& g = o->g;
    cudaStream_t q = on ? on : o->stream;
    if (mode == VSTAB_ACCUMULATED_FULL_LOCK) {
        const long anchor = lock_call - (long)o->F;
        if (o->acc_T != d_T_all || o->acc_n_total != n_total || o->acc_anchor != anchor) {
            o->err = "call vstab_offline_prepare(d_T_all, n_total, mode, lock_call) before rendering in ACCUMULATED_FULL_LOCK";
            return VSTAB_ERR_STATE;
        }
    }
    SmoothArgs a{};
    a.T = d_T_all; a.t_mod = n_total > 0 ? n_total : 1;
    a.P = (int)o->P; a.F = (int)o->F;
    a.mode = mode; a.lock_call = lock_call;
    a.acc = o->acc.as<double>(); a.acc_mod = n_total;
    a.reg = feature_lock ? o->reg_all : nullptr;
    a.reg_lo = lock_call + 1 - (long)o->F > 0 ? lock_call + 1 - (long)o->F : 0;
    a.scale = g.scale;
    a.sums = d_sums; a.sums_mod = 0; a.frame_base = frame_base;
    a.npix = (double)g.rows * (double)g.cols;
    o->timer.begin(ST_SMOOTH, q);
    launch_smooth(a, call_first, n, o->wp.as<WarpParams>(), q);
    if (o->crop.max_zoom > 1.0) {
        // the zoom of call c reads the needs of calls [c - R, c]: recompute the matrices of the calls before call_first here
        // (their presentation frames and channel sums belong to other chunks: no sums, matrices only)
        const int nhalo = (int)(call_first < o->crop.R ? call_first : o->crop.R);
        SmoothArgs ah = a;
        ah.sums = nullptr;
        launch_smooth(ah, call_first - nhalo, nhalo, o->crop_halo.as<WarpParams>(), q);
        CropArgs ca = o->crop;
        ca.rows = g.rows; ca.cols = g.cols;
        ca.need = o->crop_need.as<double>(); ca.need_base = call_first - nhalo; ca.need_mod = (long)nhalo + n;
        ca.reset = 0;
        launch_crop(ca, o->crop_halo.as<WarpParams>(), nhalo, o->wp.as<WarpParams>(), call_first, n, q);
    }
    o->timer.end(ST_SMOOTH, q);
    o->timer.begin(ST_WARP, q);
    launch_warp(d_frames, step, frame_stride, slot_mod, o->wp.as<WarpParams>(), n, g.cols, g.rows, d_out, out_step,
                out_frame_stride, q, d_check);
    o->timer.end(ST_WARP, q);
    CK(cudaGetLastError());
    o->last_ncalls = n;
    return VSTAB_OK;
}

extern "C" vstab_status vstab_offline_render(vstab_offline_t* o, const uint8_t* d_frames, size_t frame_stride,
                                              size_t step, long frame_base, int n, long call_first,
                                              const double* d_T_all, long n_total, int mode, long lock_call,
                                              const unsigned long long* d_sums,
                                              uint8_t* d_out, size_t out_frame_stride, size_t out_step) {
    return offline_render_impl(o, d_frames, frame_stride, step, frame_base, n, call_first, d_T_all, n_total, mode, lock_call,
                               d_sums, d_out, out_frame_stride, out_step, nullptr);
}

// o->acc sized for the prefix of n_total transforms (n_total matrices, then the scan's n_total / 256 + 2 block products)
static vstab_status offline_acc_reserve(vstab_offline_t* o, long n_total) {
    auto set_err = [&](const std::string& e) { o->err = e; };
    const size_t mats = (size_t)n_total + (size_t)(n_total / 256 + 2);
    if (o->acc_capacity < mats) { CK(o->acc.alloc(sizeof(double) * 9 * mats)); o->acc_capacity = mats; }
    return VSTAB_OK;
}

// vstab_offline_prepare on stream q
static vstab_status offline_prepare(vstab_offline_t* o, const double* d_T_all, long n_total, int mode, long lock_call,
                                    cudaStream_t q) {
    auto set_err = [&](const std::string& e) { o->err = e; };
    if (mode != VSTAB_ACCUMULATED_FULL_LOCK) { o->acc_T = nullptr; return VSTAB_OK; }
    if (lock_call < (long)o->F) {
        o->err = "ACCUMULATED_FULL_LOCK must be set at a call index >= future (SURVEY B.6)"; return VSTAB_ERR_STATE;
    }
    const long anchor = lock_call - (long)o->F;
    vstab_status st = offline_acc_reserve(o, n_total);
    if (st != VSTAB_OK) return st;
    o->timer.begin(ST_ACC, q);
    launch_acc_scan(d_T_all, n_total, anchor, o->acc.as<double>(), q);
    o->timer.end(ST_ACC, q);
    CK(cudaGetLastError());
    o->acc_T = d_T_all; o->acc_n_total = n_total; o->acc_anchor = anchor;
    return VSTAB_OK;
}

// The "segmented prefix/scan over 3x3 transforms" of the north star: accumulated products
// acc[k] = T[k] * ... * T[anchor+1] for the whole clip, needed by ACCUMULATED_FULL_LOCK
// (src/stabilizer.cpp:317-338).  Runs every time it is called (no caching of results).
extern "C" vstab_status vstab_offline_prepare(vstab_offline_t* o, const double* d_T_all, long n_total, int mode,
                                              long lock_call) {
    if (!o || !d_T_all || n_total < 1) return VSTAB_ERR_INVALID_ARGUMENT;
    auto set_err = [&](const std::string& e) { o->err = e; };
    CK(cudaSetDevice(o->device));
    return offline_prepare(o, d_T_all, n_total, mode, lock_call, o->stream);
}

extern "C" vstab_status vstab_offline_set_yuv(vstab_offline_t* o, const vstab_yuv_layout* in, const vstab_yuv_layout* out) {
    if (!o) return VSTAB_ERR_INVALID_ARGUMENT;
    for (const vstab_yuv_layout* L : {in, out})
        if (L && FrameFmt{true, L}.check(o->g.rows, o->g.cols, false, o->err) != VSTAB_OK) return VSTAB_ERR_INVALID_ARGUMENT;
    o->yin = in ? std::make_optional(*in) : std::nullopt;
    o->yout = out ? std::make_optional(*out) : std::nullopt;
    return VSTAB_OK;
}

extern "C" vstab_status vstab_offline_set_crop(vstab_offline_t* o, double max_zoom, double release) {
    if (!o) return VSTAB_ERR_INVALID_ARGUMENT;
    auto set_err = [&](const std::string& e) { o->err = e; };
    CropArgs c;
    if (!crop_params(max_zoom, release, &c, o->err)) return VSTAB_ERR_INVALID_ARGUMENT;
    if (c.max_zoom > 1.0) {
        CK(cudaSetDevice(o->device));
        CK(cudaStreamSynchronize(o->stream));                      // a render in flight may still read the old buffers
        CK(o->crop_halo.alloc(sizeof(WarpParams) * (size_t)c.R));
        CK(o->crop_need.alloc(sizeof(double) * ((size_t)c.R + (size_t)o->max_batch + 1)));
    }
    o->crop = c;
    return VSTAB_OK;
}

extern "C" void vstab_offline_set_timing(vstab_offline_t* o, int enable) { if (o) o->timer.enabled = enable != 0; }

// ms[8] / counts[8]: ingest, pyramid, gftt, lk, fit, smooth, warp, acc-scan since the last call
extern "C" vstab_status vstab_offline_stage_times(vstab_offline_t* o, float* ms, int* counts) {
    if (!o || !ms || !counts) return VSTAB_ERR_INVALID_ARGUMENT;
    cudaSetDevice(o->device);
    o->timer.collect(ms, counts);
    return VSTAB_OK;
}

extern "C" long long vstab_launch_count(void) { return vstabk::launch_count(); }
// VSTAB_GUARD=1: bytes found overwritten in the guard bands of released device buffers so far, and buffers checked
extern "C" vstab_status vstab_debug_link_probe(int device, const void* host_in, void* host_out, size_t bytes, size_t chunk_bytes,
                                               int passes, double* seconds) {
    auto set_err = [&](const std::string& e) { g_err = e; };
    if (!host_in || !host_out || !seconds || bytes == 0 || chunk_bytes == 0 || passes < 1) return VSTAB_ERR_INVALID_ARGUMENT;
    if (!device_ok(device, g_err)) return VSTAB_ERR_CUDA;
    DevBuf din, dout;
    cudaStream_t qi = nullptr, qo = nullptr;
    CK(din.alloc(chunk_bytes));
    CK(dout.alloc(chunk_bytes));
    CK(cudaMemset(dout.p, 0, chunk_bytes));
    CK(cudaStreamCreateWithFlags(&qi, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&qo, cudaStreamNonBlocking));
    CK(cudaDeviceSynchronize());
    const auto t0 = std::chrono::steady_clock::now();
    vstab_status st = VSTAB_OK;
    for (int p = 0; p < passes && st == VSTAB_OK; ++p)
        for (size_t o = 0; o < bytes; o += chunk_bytes) {
            const size_t n = bytes - o < chunk_bytes ? bytes - o : chunk_bytes;
            if (cudaMemcpyAsync(din.p, (const char*)host_in + o, n, cudaMemcpyHostToDevice, qi) != cudaSuccess ||
                cudaMemcpyAsync((char*)host_out + o, dout.p, n, cudaMemcpyDeviceToHost, qo) != cudaSuccess) {
                g_err = "cudaMemcpyAsync failed in the link probe"; st = VSTAB_ERR_CUDA; break;
            }
        }
    cudaStreamSynchronize(qi);
    cudaStreamSynchronize(qo);
    *seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    cudaStreamDestroy(qi);
    cudaStreamDestroy(qo);
    return st;
}

extern "C" long long vstab_debug_guard_violations(void) { return g_guard_violations.load(); }
extern "C" long long vstab_debug_guard_buffers(void) { return g_guard_buffers.load(); }

extern "C" long vstab_offline_read_h(vstab_offline_t* o, double* dst, size_t n_calls) {
    if (!o || !dst) return -1;
    if (cudaSetDevice(o->device) != cudaSuccess) return -1;
    if (cudaStreamSynchronize(o->stream) != cudaSuccess) return -1;
    size_t n = n_calls < (size_t)o->last_ncalls ? n_calls : (size_t)o->last_ncalls;
    std::vector<WarpParams> h(n);
    if (n && cudaMemcpy(h.data(), o->wp.p, sizeof(WarpParams) * n, cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
    for (size_t i = 0; i < n; ++i) memcpy(dst + i * 9, h[i].Hs, sizeof(double) * 9);
    return (long)n;
}

// =====================================================================================
// sharded offline job: NCCL (resolved at run time) + vstab_offline_run
// =====================================================================================
// NCCL is bound with dlopen so that single-GPU users of libvstab.so need no NCCL at all and a host process that already
// carries one (torch's bundled libnccl.so.2) shares it.  Only the six entry points below are used; their signatures are
// those of nccl.h 2.x (ncclResult_t = int, ncclDataType_t: ncclUint8 = 1, ncclDouble = 8).
static void poses_to_render(const double* poses, long n, RenderPose* hp);
namespace {
struct NcclApi {
    void* lib = nullptr;
    int (*GetUniqueId)(void*) = nullptr;
    int (*CommInitRank)(void**, int, vstab_nccl_id, int) = nullptr;     // ncclUniqueId is a 128-byte struct passed by value
    int (*CommDestroy)(void*) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
    int (*Broadcast)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
    std::string err;
    bool load() {
        if (lib) return true;
        const char* names[] = {"libnccl.so.2", "libnccl.so"};
        for (const char* n : names) { lib = dlopen(n, RTLD_NOW | RTLD_NOLOAD | RTLD_GLOBAL); if (lib) break; }   // one already in the process
        if (!lib) for (const char* n : names) { lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL); if (lib) break; }
        if (!lib) { err = std::string("NCCL not found (dlopen libnccl.so.2): ") + (dlerror() ? dlerror() : ""); return false; }
        auto sym = [&](const char* n) { void* p = dlsym(lib, n); if (!p) err = std::string("NCCL symbol missing: ") + n; return p; };
        GetUniqueId = (decltype(GetUniqueId))sym("ncclGetUniqueId");
        CommInitRank = (decltype(CommInitRank))sym("ncclCommInitRank");
        CommDestroy = (decltype(CommDestroy))sym("ncclCommDestroy");
        AllGather = (decltype(AllGather))sym("ncclAllGather");
        Broadcast = (decltype(Broadcast))sym("ncclBroadcast");
        GetErrorString = (decltype(GetErrorString))sym("ncclGetErrorString");
        if (!GetUniqueId || !CommInitRank || !CommDestroy || !AllGather || !Broadcast || !GetErrorString) { lib = nullptr; return false; }
        return true;
    }
};
NcclApi g_nccl;
std::mutex g_nccl_mu;
constexpr int kNcclUint8 = 1, kNcclDouble = 8;

// Device time of the phases of one vstab_offline_run, and the events that order its streams.  Spans are recorded only when a
// report is asked for (`on`), and only spans carry timestamps: timed events between the copies of a copy stream left the
// link idle for ~200 us per 16-frame chunk instead of ~50 (1080p run_host, B200 at 1000 W).
struct PhaseClock {
    bool on = false;
    std::vector<std::pair<int, std::pair<cudaEvent_t, cudaEvent_t>>> spans;
    std::vector<cudaEvent_t> pool;
    cudaEvent_t get(bool timed = false) {
        cudaEvent_t e = nullptr;
        cudaEventCreateWithFlags(&e, timed ? cudaEventDefault : cudaEventDisableTiming);
        pool.push_back(e);
        return e;
    }
    void begin(int phase, cudaStream_t q) { if (!on) return; cudaEvent_t e = get(true); cudaEventRecord(e, q); spans.push_back({phase, {e, nullptr}}); }
    void end(cudaStream_t q) { if (!on) return; cudaEvent_t e = get(true); cudaEventRecord(e, q); spans.back().second.second = e; }
    void collect(float* ms4) {
        for (auto& sp : spans) { float ms = 0.f; if (sp.second.second && cudaEventElapsedTime(&ms, sp.second.first, sp.second.second) == cudaSuccess) ms4[sp.first] += ms; }
    }
    ~PhaseClock() { for (auto e : pool) cudaEventDestroy(e); }
};
}  // namespace

namespace { void nccl_comm_destroy(void* comm) { if (comm && g_nccl.CommDestroy) g_nccl.CommDestroy(comm); } }

extern "C" const char* vstab_offline_last_error(const vstab_offline_t* o) { return o ? o->err.c_str() : g_err.c_str(); }

extern "C" vstab_status vstab_nccl_get_unique_id(vstab_nccl_id* out) {
    if (!out) return VSTAB_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(g_nccl_mu);
    if (!g_nccl.load()) { g_err = g_nccl.err; return VSTAB_ERR_NCCL; }
    const int r = g_nccl.GetUniqueId(out);
    if (r != 0) { g_err = std::string("ncclGetUniqueId: ") + g_nccl.GetErrorString(r); return VSTAB_ERR_NCCL; }
    return VSTAB_OK;
}

extern "C" vstab_status vstab_offline_comm_init(vstab_offline_t* o, const vstab_nccl_id* id, int rank, int world) {
    if (!o || !id || world < 1 || rank < 0 || rank >= world) return VSTAB_ERR_INVALID_ARGUMENT;
    auto set_err = [&](const std::string& e) { o->err = e; };
    {
        std::lock_guard<std::mutex> lock(g_nccl_mu);
        if (!g_nccl.load()) { o->err = g_nccl.err; return VSTAB_ERR_NCCL; }
    }
    CK(cudaSetDevice(o->device));
    if (o->comm) { g_nccl.CommDestroy(o->comm); o->comm = nullptr; }
    const int r = g_nccl.CommInitRank(&o->comm, world, *id, rank);
    if (r != 0) { o->comm = nullptr; o->err = std::string("ncclCommInitRank: ") + g_nccl.GetErrorString(r); return VSTAB_ERR_NCCL; }
    o->rank = rank; o->world = world;
    // NCCL connects the ranks lazily, inside the first collective (~1.5 s on an 8-GPU NVSwitch box): pay for it here, with
    // one 8-byte all-gather, instead of inside the first job
    DevBuf warm;
    CK(warm.alloc(sizeof(double) * (size_t)(world + 1)));
    CK(cudaMemsetAsync(warm.p, 0, sizeof(double) * (size_t)(world + 1), o->stream));
    const int rw = g_nccl.AllGather(warm.as<double>() + world, warm.p, 1, kNcclDouble, o->comm, o->stream);
    if (rw != 0) { o->err = std::string("ncclAllGather (warm-up): ") + g_nccl.GetErrorString(rw); return VSTAB_ERR_NCCL; }
    CK(cudaStreamSynchronize(o->stream));
    return VSTAB_OK;
}

extern "C" vstab_status vstab_offline_plan(long n_total, int world, int rank, size_t future_frames, vstab_shard_plan* out) {
    if (!out || n_total < 1 || world < 1 || rank < 0 || rank >= world) return VSTAB_ERR_INVALID_ARGUMENT;
    const long base = n_total / world, rem = n_total % world;
    const long first = rank * base + (rank < rem ? rank : rem);
    const long last = first + base + (rank < rem ? 1 : 0);
    out->first = first; out->last = last;
    if (last <= first) { out->call_first = out->call_last = 0; return VSTAB_OK; }
    const long F = (long)future_frames;
    const long c0 = first == 0 ? 0 : first + F;
    const long c1 = last + F < n_total ? last + F : n_total;
    out->call_first = c0; out->call_last = c1 > c0 ? c1 : c0;
    return VSTAB_OK;
}

extern "C" vstab_status vstab_offline_fused_plan(long n_total, int world, int rank, size_t past_frames, size_t future_frames,
                                                 int max_batch, vstab_fused_plan* out) {
    vstab_shard_plan pl;
    if (!out || max_batch < 1) return VSTAB_ERR_INVALID_ARGUMENT;
    const vstab_status st = vstab_offline_plan(n_total, world, rank, future_frames, &pl);
    if (st != VSTAB_OK) return st;
    const long P = (long)past_frames, F = (long)future_frames, B = max_batch;
    out->ring_chunks = (F > 1 ? (F - 1 + B - 1) / B : 0) + 3;      // lag of the warp step + 2 for the three streams
    // first call whose window starts inside the rank's own transforms T[first ..] (rank 0: T[0] is never read)
    long head = pl.call_first;
    if (pl.first > 0 && pl.first + P + F - 1 > head) head = pl.first + P + F - 1;
    if (head > pl.call_last) head = pl.call_last;
    // call c reads transforms up to T[c - 1]: the last one the rank estimates itself is T[last - 1]
    long tail = pl.last + 1 < pl.call_last ? pl.last + 1 : pl.call_last;
    if (tail < head) tail = head;
    out->fused_first = head; out->fused_last = tail;
    return VSTAB_OK;
}

extern "C" uint64_t vstab_frame_checksum(const uint8_t* bgr, int rows, int cols, size_t step) {
    uint64_t sum = 0;
    const int groups = (cols + 3) / 4;
    for (int y = 0; y < rows; ++y) {
        const uint8_t* row = bgr + (size_t)y * step;
        for (int g = 0; g < groups; ++g) {
            uint8_t b[12] = {0};
            const int nb = 3 * ((cols - 4 * g) < 4 ? (cols - 4 * g) : 4);
            memcpy(b, row + (size_t)12 * g, (size_t)nb);
            uint32_t w[3];
            for (int k = 0; k < 3; ++k) w[k] = (uint32_t)b[4 * k] | ((uint32_t)b[4 * k + 1] << 8) | ((uint32_t)b[4 * k + 2] << 16) | ((uint32_t)b[4 * k + 3] << 24);
            sum += (uint64_t)(y + 1) * (uint64_t)(g + 1) * ((uint64_t)w[0] + 3ull * w[1] + 5ull * w[2]);
        }
    }
    return sum;
}

// vstab_offline_run as rank `rank` of a world of `world` ranks (the instance's communicator carries the exchange when world > 1)
static vstab_status offline_job(vstab_offline_t* o, const vstab_offline_cfg* cfg, vstab_offline_report* rep, int world, int rank) {
    if (!o || !cfg || cfg->n_total < 1) return VSTAB_ERR_INVALID_ARGUMENT;
    auto set_err = [&](const std::string& e) { o->err = e; };
    Geometry& g = o->g;
    const long N = cfg->n_total;
    const int mode = cfg->mode;
    const bool sim = cfg->source == VSTAB_SRC_SIMULATOR;
    // caller frames (the simulator's frames are the library's own) and the sink of the outputs, if any
    const FrameFmt in{cfg->source != VSTAB_SRC_DEVICE, o->yin && !sim ? &*o->yin : nullptr, cfg->step, cfg->frame_stride};
    const FrameFmt out{cfg->host_out != nullptr, o->yout ? &*o->yout : nullptr, cfg->out_step, cfg->out_frame_stride};
    uint8_t* const sink = cfg->d_out ? cfg->d_out : cfg->host_out;
    // a device BGR shard is read where it is; a YUV device shard is staged through the chunk ring like a host one
    // (converted instead of copied)
    const bool resident = in.direct();
    const bool direct = sink && out.direct();                      // the warp writes the caller's BGR buffer itself
    const bool feature_lock = mode == VSTAB_ORB_FULL_LOCK || mode == VSTAB_SIFT_FULL_LOCK;
    if (mode < 0 || mode > 5) { o->err = "Stabilizer: Invalid stabilization mode"; return VSTAB_ERR_INVALID_ARGUMENT; }
    if (sim && (!cfg->d_texture || !cfg->poses || cfg->tex_rows < 1 || cfg->tex_cols < 1)) { o->err = "simulator source needs d_texture and poses"; return VSTAB_ERR_INVALID_ARGUMENT; }
    const char* src_err = "host / device source needs frames with step >= 3*cols";
    if (!sim && !cfg->host_frames) { o->err = src_err; return VSTAB_ERR_INVALID_ARGUMENT; }
    vstab_status st = sim ? VSTAB_OK : in.check(g.rows, g.cols, true, o->err, src_err);
    if (st == VSTAB_OK && sink) st = out.check(g.rows, g.cols, true, o->err, "out_step smaller than 3*cols");
    if (st != VSTAB_OK) return st;
    if (cfg->host_out && cfg->d_out) { o->err = "give host_out or d_out, not both"; return VSTAB_ERR_INVALID_ARGUMENT; }
    if ((mode == VSTAB_ACCUMULATED_FULL_LOCK || feature_lock) && cfg->lock_call < (long)o->F) {
        o->err = "lock modes must be set at a call index >= future (SURVEY B.6)"; return VSTAB_ERR_STATE;
    }
    CK(cudaSetDevice(o->device));
    vstab_shard_plan pl;
    vstab_offline_plan(N, world, rank, o->F, &pl);
    if (!sim && pl.first > 0 && !cfg->host_halo) { o->err = "host source: host_halo (frame first-1) required on ranks > 0"; return VSTAB_ERR_INVALID_ARGUMENT; }
    const long n_local = pl.last - pl.first, n_calls = pl.call_last - pl.call_first;
    const long L = (N + world - 1) / world;                        // padded shard length of the all-gather
    const int B = o->max_batch;
    const long F = (long)o->F;
    cudaStream_t q = o->stream;
    PhaseClock clock;
    clock.on = rep != nullptr;
    enum { PH_SOURCE = 0, PH_ESTIMATE = 1, PH_EXCHANGE = 2, PH_RENDER = 3 };

    // ---- buffers: one chunk of frames (+ halo), one or two chunks of outputs, transforms, sums, checksums -------------
    // GLOBAL_SMOOTHING from a staged source (simulator, host) is ONE pass: the window of call c reads T[c-P-F+1 .. c-1] and
    // nothing else, so the calls whose windows are complete are warped right behind the estimation, from a ring of the last
    // ceil((F-1)/B) + 3 chunks -- every frame is rendered / uploaded once instead of twice.  The calls whose windows reach
    // into a neighbour's shard (the first P-1 and the last F-1 of a rank in a world > 1) wait for the all-gather as before.
    // In a world of one every LK-path mode is one pass: the lock modes read the prefix of the transforms estimated so far
    // (ACCUMULATED_FULL_LOCK) or nothing at all (TRANSLATION_LOCK / ROTATION_LOCK).
    const bool fused = !resident && (mode == VSTAB_GLOBAL_SMOOTHING || (world == 1 && !feature_lock));
    vstab_fused_plan fp;
    // with auto-crop the matrices of call c come from the windows of calls c - R .. c: a window of past P + R
    vstab_offline_fused_plan(N, world, rank, o->P + (size_t)o->crop.R, o->F, B, &fp);
    const long ring_chunks = fused ? fp.ring_chunks : 1;
    const long ring_frames = ring_chunks * B;                       // + one slot for the halo frame of the first chunk
    // outputs for a host sink leave on a download stream of their own, out of two halves of the output chunk (and of the
    // YUV staging): batch i is warped and converted into half i % 2 while the download of batch i - 1 reads the other one
    const bool split = cfg->host_out != nullptr;
    const int halves = split ? 2 : 1;
    DevBuf& chunk = o->job_chunk; DevBuf& outc = o->job_out;
    if (!(resident && direct) && o->job_chunk_frames < (size_t)ring_frames + 1) {
        CK(chunk.alloc(g.frame_bytes * ((size_t)ring_frames + 1) + 64));
        o->job_chunk_frames = (size_t)ring_frames + 1;
    }
    if (!(resident && direct) && o->job_out_frames < (size_t)B * halves) {
        CK(outc.alloc(g.frame_bytes * (size_t)B * halves + 64));
        o->job_out_frames = (size_t)B * halves;
    }
    DevBuf T_local, T_gather, T_all, sums, checks, poses_d, rays_d, tex4_d, reg_local, reg_gather, reg_all;
    CK(T_local.alloc(sizeof(double) * 9 * (size_t)L));
    CK(T_all.alloc(sizeof(double) * 9 * (size_t)N));
    if (world > 1) CK(T_gather.alloc(sizeof(double) * 9 * (size_t)L * world));
    CK(sums.alloc(sizeof(unsigned long long) * 3 * (size_t)(n_local > 0 ? n_local : 1)));
    CK(checks.alloc(sizeof(unsigned long long) * (size_t)(n_calls > 0 ? n_calls : 1)));
    CK(cudaMemsetAsync(T_local.p, 0, sizeof(double) * 9 * (size_t)L, q));
    CK(cudaMemsetAsync(checks.p, 0, sizeof(unsigned long long) * (size_t)(n_calls > 0 ? n_calls : 1), q));
    uint8_t* cb = chunk.as<uint8_t>();
    const size_t fb = g.frame_bytes;
    // staging of host YUV frames: B frames for the fetches on q, two halves of B frames for the source stream of the fused
    // pass (chunk k uploads into half k % 2, q converts it before E(k), and S(k+2) waits for E(k)), and one download
    // staging per output half
    const size_t istage = in.staging_bytes(g) * (size_t)B, ostage = out.staging_bytes(g) * (size_t)B;
    if (o->job_stage_bytes < 3 * istage + halves * ostage) {
        CK(o->job_stage.alloc(3 * istage + halves * ostage));
        o->job_stage_bytes = 3 * istage + halves * ostage;
    }
    uint8_t* const ystage_q = o->job_stage.as<uint8_t>();
    uint8_t* const ystage_qs = ystage_q + istage;
    uint8_t* const ystage_o = ystage_qs + 2 * istage;
    // caller frame f of the clip (host or device memory); a resident shard is read there, with no staging
    auto dframe = [&](long f) -> const uint8_t* { return f == pl.first - 1 ? cfg->host_halo : cfg->host_frames + (size_t)(f - pl.first) * cfg->frame_stride; };
    const size_t src_fs = resident ? cfg->frame_stride : fb, src_step = resident ? cfg->step : g.pitch;
    // simulator: poses of the frames this rank may touch (first-1 .. last-1, the anchor frame), as renderer poses
    if (sim) {
        std::vector<RenderPose> hp((size_t)N);
        poses_to_render(cfg->poses, N, hp.data());                  // all N (72 + 24 bytes each): the anchor frame may be anyone's
        CK(poses_d.alloc(sizeof(RenderPose) * (size_t)N));
        CK(cudaMemcpyAsync(poses_d.p, hp.data(), sizeof(RenderPose) * (size_t)N, cudaMemcpyHostToDevice, q));
        // the camera rays do not depend on the pose: once per job (24 bytes per pixel), not once per pixel and frame
        CK(rays_d.alloc(sizeof(double) * 3 * (size_t)g.cols * g.rows));
        launch_render_rays(g.cols, g.rows, cfg->focal, rays_d.as<double>(), q);
        CK(tex4_d.alloc(sizeof(unsigned) * (size_t)cfg->tex_rows * cfg->tex_cols));
        launch_render_tex4(cfg->d_texture, cfg->tex_rows, cfg->tex_cols, tex4_d.as<unsigned>(), q);
        CK(cudaStreamSynchronize(q));                               // hp goes out of scope
    }
    // frames [f0, f0 + n) of the clip -> chunk slots [slot, slot + n) on stream q, caller frames through the staging `stg`;
    // convert = false leaves the conversion of YUV frames (frames_in_convert) to the caller
    auto fetch = [&](long f0, long n, int slot, cudaStream_t q, uint8_t* stg, bool convert = true) -> vstab_status {
        if (n <= 0 || resident) return VSTAB_OK;
        clock.begin(PH_SOURCE, q);
        if (sim) {
            launch_render(cfg->d_texture, cfg->tex_rows, cfg->tex_cols, poses_d.as<RenderPose>() + f0, (int)n, g.cols, g.rows, cfg->focal,
                          cb + (size_t)slot * fb, g.pitch, fb, q, rays_d.as<double>(), tex4_d.as<unsigned>());
        } else {
            if (f0 < pl.first - 1 || f0 + n > pl.last) { o->err = "internal: frame outside the rank's shard"; return VSTAB_ERR_STATE; }
            for (long i = 0; i < n;) {
                const long f = f0 + i;
                const long m = f == pl.first - 1 ? 1 : n - i;      // the halo frame alone, then one contiguous run
                uint8_t* dst = cb + (size_t)(slot + i) * fb;
                uint8_t* st = stg + (size_t)i * in.staging_bytes(g);
                CK(frames_in_transfer(g, in, dframe(f), m, dst, st, q));
                if (convert) CK(frames_in_convert(g, in, dframe(f), m, dst, st, q));
                i += m;
            }
        }
        clock.end(q);
        CK(cudaGetLastError());
        return VSTAB_OK;
    };
    cudaEvent_t ev_t0 = clock.get(true), ev_t1 = clock.get(true);
    CK(cudaEventRecord(ev_t0, q));

    // ---- ORB / SIFT lock: reference set from the anchor frame, broadcast from its owner --------------------------
    if (feature_lock) {
        const long anchor = cfg->lock_call - F > 0 ? cfg->lock_call - F : 0;       // presentation frame of the call that set the mode
        int owner = 0;
        for (int r = 0; r < world; ++r) { vstab_shard_plan q2; vstab_offline_plan(N, world, r, o->F, &q2); if (anchor >= q2.first && anchor < q2.last) owner = r; }
        st = offline_feature_setup(o, mode);
        if (st != VSTAB_OK) return st;
        DevBuf pack;
        CK(pack.alloc(vstab_offline_reference_bytes()));
        if (rank == owner) {
            if ((st = fetch(anchor, 1, 0, q, ystage_q)) != VSTAB_OK) return st;
            if ((st = vstab_offline_reference_capture(o, resident ? dframe(anchor) : cb, src_step, mode)) != VSTAB_OK) return st;
            if ((st = vstab_offline_reference_export(o, pack.p)) != VSTAB_OK) return st;
        }
        if (world > 1) {
            clock.begin(PH_EXCHANGE, q);
            const int r = g_nccl.Broadcast(pack.p, pack.p, vstab_offline_reference_bytes(), kNcclUint8, owner, o->comm, q);
            clock.end(q);
            if (r != 0) { o->err = std::string("ncclBroadcast: ") + g_nccl.GetErrorString(r); return VSTAB_ERR_NCCL; }
            if (rank != owner && (st = vstab_offline_reference_import(o, pack.p, mode)) != VSTAB_OK) return st;
        }
        CK(cudaStreamSynchronize(q));                               // `pack` is released here
        CK(reg_local.alloc(sizeof(double) * 10 * (size_t)L));
        CK(reg_all.alloc(sizeof(double) * 10 * (size_t)N));
        if (world > 1) CK(reg_gather.alloc(sizeof(double) * 10 * (size_t)L * world));
        CK(cudaMemsetAsync(reg_local.p, 0, sizeof(double) * 10 * (size_t)L, q));
    }

    if (split && !o->download) CK(cudaStreamCreateWithFlags(&o->download, cudaStreamNonBlocking));
    cudaEvent_t ev_warped = clock.get(), ev_down[2] = {clock.get(), clock.get()};
    long batches = 0;                                               // batches warped so far
    // warps the calls [c0, c1) (at most B per launch) on stream qw, in mode `rmode` over the transforms T_all[0 .. nT);
    // ring > 0: their presentation frames are in the ring already
    auto render_calls = [&](long c0, long c1, long ring, int rmode, long nT, cudaStream_t qw) -> vstab_status {
        for (long c = c0; c < c1; c += B, ++batches) {
            const long n = c1 - c < B ? c1 - c : B;
            const long p_lo = c - F > 0 ? c - F : 0, p_hi = c + n - 1 - F > 0 ? c + n - 1 - F : 0;
            vstab_status s2;
            if (ring == 0 && (s2 = fetch(p_lo, p_hi - p_lo + 1, 0, qw, ystage_q)) != VSTAB_OK) return s2;
            const int h = (int)(batches % halves);
            if (split && batches >= 2) CK(cudaStreamWaitEvent(qw, ev_down[h], 0));   // the download of batch - 2 read half h
            uint8_t* ob = outc.as<uint8_t>() + (size_t)h * B * fb;
            uint8_t* stg = ystage_o + (size_t)h * ostage;
            clock.begin(PH_RENDER, qw);
            uint8_t* dst = direct ? cfg->d_out + (size_t)(c - pl.call_first) * cfg->out_frame_stride : ob;
            const long base = ring > 0 ? pl.first : p_lo;          // frame held by slot 0 (ring: modulo `ring`)
            s2 = offline_render_impl(o, resident ? dframe(p_lo) : cb, src_fs, src_step, base, (int)n, c, T_all.as<double>(), nT, rmode,
                                     cfg->lock_call, sums.as<unsigned long long>() + (size_t)(base - pl.first) * 3, dst,
                                     direct ? cfg->out_frame_stride : fb, direct ? cfg->out_step : g.pitch,
                                     cfg->checksums ? checks.as<unsigned long long>() + (c - pl.call_first) : nullptr, ring, qw);
            clock.end(qw);
            if (s2 != VSTAB_OK) return s2;
            if (sink && !direct) {
                uint8_t* to = sink + (size_t)(c - pl.call_first) * cfg->out_frame_stride;
                CK(frames_out_convert(g, out, ob, n, to, stg, qw));
                if (split) {
                    CK(cudaEventRecord(ev_warped, qw));
                    CK(cudaStreamWaitEvent(o->download, ev_warped, 0));
                }
                CK(frames_out_transfer(g, out, ob, n, to, stg, split ? o->download : qw));
                if (split) CK(cudaEventRecord(ev_down[h], o->download));
            }
        }
        return VSTAB_OK;
    };
    // calls [call_first, c_head) and [c_tail, call_last) are warped after the exchange; the fused pass serves the rest
    long c_head = pl.call_first, c_tail = pl.call_first;

    // ---- fused pass: estimate chunk k, then warp every call whose window is complete -----------------------------------
    // Three streams, so that the source (f64 rendering, or PCIe uploads), the estimation and the warps of neighbouring chunks
    // overlap -- they load different pipes of the SM: source of chunk k+1, k+2 (qs) || estimate k (q) || warp step k-1 (qw).
    // Chunk j is written by S(j) and read by E(j), E(j+1) (halo) and the warp steps W(j) .. W(j + lag); S(j) overwrites
    // chunk j - ring_chunks, so it waits for W(j-3) (lag = ring_chunks - 3) and E(j-2).
    if (fused) {
        if (!o->copy_in) CK(cudaStreamCreateWithFlags(&o->copy_in, cudaStreamNonBlocking));
        if (!o->copy_out) CK(cudaStreamCreateWithFlags(&o->copy_out, cudaStreamNonBlocking));
        cudaStream_t qs = o->copy_in, qw = o->copy_out;
        constexpr int kEv = 8;
        cudaEvent_t evS[kEv], evE[kEv], evW[kEv];
        for (int i = 0; i < kEv; ++i) { evS[i] = clock.get(); evE[i] = clock.get(); evW[i] = clock.get(); }
        CK(cudaMemsetAsync(T_all.p, 0, sizeof(double) * 9 * (size_t)N, q));
        if (mode == VSTAB_ACCUMULATED_FULL_LOCK && (st = offline_acc_reserve(o, N)) != VSTAB_OK) return st;   // no reallocation in flight
        cudaEvent_t ev_ready = clock.get();                        // the job's buffers are reset (q) before qs / qw touch them
        CK(cudaEventRecord(ev_ready, q));
        CK(cudaStreamWaitEvent(qs, ev_ready, 0));
        CK(cudaStreamWaitEvent(qw, ev_ready, 0));
        c_head = c_tail = fp.fused_first;
        const long nchunks = (n_local + B - 1) / B;
        auto stg_qs = [&](long k) { return ystage_qs + (size_t)(k % 2) * istage; };
        auto source = [&](long k) -> vstab_status {               // S(k)
            const long f0 = pl.first + k * B, n = pl.last - f0 < B ? pl.last - f0 : B;
            if (k >= 3) CK(cudaStreamWaitEvent(qs, evW[(k - 3) % kEv], 0));
            if (k >= 2) CK(cudaStreamWaitEvent(qs, evE[(k - 2) % kEv], 0));
            vstab_status s2;
            if (k == 0 && f0 > 0 && (s2 = fetch(f0 - 1, 1, (int)ring_frames, qs, stg_qs(k))) != VSTAB_OK) return s2;
            if ((s2 = fetch(f0, n, (int)((k % ring_chunks) * B), qs, stg_qs(k), false)) != VSTAB_OK) return s2;
            CK(cudaEventRecord(evS[k % kEv], qs));
            return VSTAB_OK;
        };
        if (nchunks > 0 && (st = source(0)) != VSTAB_OK) return st;
        if (nchunks > 1 && (st = source(1)) != VSTAB_OK) return st;
        for (long k = 0; k < nchunks; ++k) {
            const long f0 = pl.first + k * B, n = pl.last - f0 < B ? pl.last - f0 : B;
            const long slot0 = (k % ring_chunks) * B;
            const uint8_t* hl = nullptr;
            if (k == 0) { if (f0 > 0) hl = cb + (size_t)ring_frames * fb; }
            else hl = cb + (size_t)(((k - 1) % ring_chunks) * B + B - 1) * fb;      // the previous chunk's last frame, still in the ring
            CK(cudaStreamWaitEvent(q, evS[k % kEv], 0));
            if (in.yuv) {                                           // YUV frames staged (or left in place) by S(k)
                clock.begin(PH_SOURCE, q);
                CK(frames_in_convert(g, in, dframe(f0), n, cb + (size_t)slot0 * fb, stg_qs(k), q));
                clock.end(q);
            }
            clock.begin(PH_ESTIMATE, q);
            st = vstab_offline_estimate(o, cb + (size_t)slot0 * fb, src_fs, src_step, (int)n, f0, hl, T_all.as<double>() + (size_t)f0 * 9,
                                        sums.as<unsigned long long>() + (size_t)(f0 - pl.first) * 3);
            clock.end(q);
            if (st != VSTAB_OK) return st;
            CK(cudaEventRecord(evE[k % kEv], q));
            if (k + 2 < nchunks && (st = source(k + 2)) != VSTAB_OK) return st;
            // W(k): call c reads transforms up to T[c - 1] and presents frame c - F (future 0: T[c] and frame c)
            CK(cudaStreamWaitEvent(qw, evE[k % kEv], 0));
            const long c_end = f0 + n + (F > 0 ? 1 : 0);
            const long c_ok = c_end < fp.fused_last ? c_end : fp.fused_last;
            if (c_ok > c_tail) {
                const long p_lo = c_tail - F > 0 ? c_tail - F : 0;
                if (p_lo < pl.first || p_lo - pl.first < (k - (ring_chunks - 3)) * B) { o->err = "internal: presentation frame left the ring"; return VSTAB_ERR_STATE; }
                // ACCUMULATED_FULL_LOCK (world of one): the prefix over the frames estimated so far, rescanned on qw because
                // W(k-1) reads the one it replaces; until the anchor frame is in, every call is before the lock call
                int rmode = mode;
                const long seen = f0 + n, nT = mode == VSTAB_ACCUMULATED_FULL_LOCK ? seen : N;
                if (mode == VSTAB_ACCUMULATED_FULL_LOCK) {
                    if (seen <= cfg->lock_call - F) rmode = VSTAB_GLOBAL_SMOOTHING;
                    else if ((st = offline_prepare(o, T_all.as<double>(), seen, mode, cfg->lock_call, qw)) != VSTAB_OK) return st;
                }
                if ((st = render_calls(c_tail, c_ok, ring_frames, rmode, nT, qw)) != VSTAB_OK) return st;
                c_tail = c_ok;
            }
            CK(cudaEventRecord(evW[k % kEv], qw));
        }
        if (nchunks > 0) CK(cudaStreamWaitEvent(q, evW[(nchunks - 1) % kEv], 0));
        if (c_tail != fp.fused_last) { o->err = "internal: the fused pass did not reach its last call"; return VSTAB_ERR_STATE; }
        if (n_local > 0)
            CK(cudaMemcpyAsync(T_local.p, T_all.as<double>() + (size_t)pl.first * 9, sizeof(double) * 9 * (size_t)n_local, cudaMemcpyDeviceToDevice, q));
    }

    // ---- pass 1: estimate T[f] for f in [first, last), chunk by chunk ----------------------------------------------
    for (long f0 = pl.first; f0 < pl.last && !fused; f0 += B) {
        const long n = pl.last - f0 < B ? pl.last - f0 : B;
        if (!resident) {
            if (f0 == pl.first) {
                if (f0 > 0 && (st = fetch(f0 - 1, 1, 0, q, ystage_q)) != VSTAB_OK) return st;     // halo frame
            } else {
                // the last frame of the previous chunk is this chunk's halo
                CK(cudaMemcpyAsync(cb, cb + (size_t)B * fb, fb, cudaMemcpyDeviceToDevice, q));
            }
            if ((st = fetch(f0, n, 1, q, ystage_q)) != VSTAB_OK) return st;
        }
        const uint8_t* fr = resident ? dframe(f0) : cb + fb;
        const uint8_t* hl = f0 > 0 ? (resident ? dframe(f0 - 1) : cb) : nullptr;
        clock.begin(PH_ESTIMATE, q);
        st = vstab_offline_estimate(o, fr, src_fs, src_step, (int)n, f0, hl,
                                    T_local.as<double>() + (size_t)(f0 - pl.first) * 9,
                                    sums.as<unsigned long long>() + (size_t)(f0 - pl.first) * 3);
        if (st == VSTAB_OK && feature_lock)
            st = vstab_offline_register(o, fr, src_fs, src_step, (int)n, reg_local.as<double>() + (size_t)(f0 - pl.first) * 10);
        clock.end(q);
        if (st != VSTAB_OK) return st;
    }

    // ---- the exchange: one all-gather of 72 bytes per frame (+ 80 bytes per frame of registrations) ----------------
    clock.begin(PH_EXCHANGE, q);
    auto gather = [&](DevBuf& local, DevBuf& gathered, DevBuf& all, size_t per_frame) -> vstab_status {
        if (world == 1) {
            CK(cudaMemcpyAsync(all.p, local.p, sizeof(double) * per_frame * (size_t)N, cudaMemcpyDeviceToDevice, q));
            return VSTAB_OK;
        }
        const int r = g_nccl.AllGather(local.p, gathered.p, per_frame * (size_t)L, kNcclDouble, o->comm, q);
        if (r != 0) { o->err = std::string("ncclAllGather: ") + g_nccl.GetErrorString(r); return VSTAB_ERR_NCCL; }
        for (int rr = 0; rr < world; ++rr) {                       // drop the padding of the shorter shards
            vstab_shard_plan q2; vstab_offline_plan(N, world, rr, o->F, &q2);
            if (q2.last > q2.first)
                CK(cudaMemcpyAsync(all.as<double>() + (size_t)q2.first * per_frame, gathered.as<double>() + (size_t)rr * L * per_frame,
                                   sizeof(double) * per_frame * (size_t)(q2.last - q2.first), cudaMemcpyDeviceToDevice, q));
        }
        return VSTAB_OK;
    };
    if ((st = gather(T_local, T_gather, T_all, 9)) != VSTAB_OK) return st;
    if (feature_lock) {
        if ((st = gather(reg_local, reg_gather, reg_all, 10)) != VSTAB_OK) return st;
        if ((st = vstab_offline_set_registrations(o, reg_all.as<double>(), N)) != VSTAB_OK) return st;
    }
    const bool pass2 = c_head > pl.call_first || c_tail < pl.call_last;
    if (pass2 && (st = offline_prepare(o, T_all.as<double>(), N, mode, cfg->lock_call, q)) != VSTAB_OK) return st;
    clock.end(q);

    // ---- pass 2: the calls whose presentation frame this rank owns (all of them, or what the fused pass left) ----------
    if ((st = render_calls(pl.call_first, c_head, 0, mode, N, q)) != VSTAB_OK) return st;
    if ((st = render_calls(c_tail, pl.call_last, 0, mode, N, q)) != VSTAB_OK) return st;
    if (split && batches > 0) CK(cudaStreamWaitEvent(q, ev_down[(batches - 1) % 2], 0));
    if (cfg->checksums && n_calls > 0)
        CK(cudaMemcpyAsync(cfg->checksums, checks.p, sizeof(unsigned long long) * (size_t)n_calls, cudaMemcpyDeviceToHost, q));
    if (cfg->T_all) CK(cudaMemcpyAsync(cfg->T_all, T_all.p, sizeof(double) * 9 * (size_t)N, cudaMemcpyDeviceToHost, q));
    CK(cudaEventRecord(ev_t1, q));
    CK(cudaStreamSynchronize(q));
    o->acc_T = nullptr;                                            // T_all dies with this call
    o->reg_all = nullptr; o->reg_n = 0;
    if (rep) {
        float ms[4] = {0, 0, 0, 0};
        clock.collect(ms);
        rep->source_ms = ms[PH_SOURCE]; rep->estimate_ms = ms[PH_ESTIMATE]; rep->exchange_ms = ms[PH_EXCHANGE]; rep->render_ms = ms[PH_RENDER];
        rep->total_ms = 0.f;
        cudaEventElapsedTime(&rep->total_ms, ev_t0, ev_t1);
        rep->frames = n_local; rep->calls = n_calls;
    }
    CK(cudaGetLastError());
    return VSTAB_OK;
}

extern "C" vstab_status vstab_offline_run(vstab_offline_t* o, const vstab_offline_cfg* cfg, vstab_offline_report* rep) {
    if (!o) return VSTAB_ERR_INVALID_ARGUMENT;
    return offline_job(o, cfg, rep, o->comm ? o->world : 1, o->comm ? o->rank : 0);
}

// the job of vstab_offline_run in a world of one (whatever communicator the instance has joined), host frames in and out
extern "C" vstab_status vstab_offline_run_host(vstab_offline_t* o, const uint8_t* frames, size_t frame_stride, size_t step,
                                                long n_total, int mode, long lock_call, uint8_t* out,
                                                size_t out_frame_stride, size_t out_step) {
    if (!o || !frames || !out || n_total < 1) return VSTAB_ERR_INVALID_ARGUMENT;
    vstab_offline_cfg cfg{};
    cfg.n_total = n_total; cfg.mode = mode; cfg.lock_call = lock_call; cfg.source = VSTAB_SRC_HOST;
    cfg.host_frames = frames; cfg.frame_stride = frame_stride; cfg.step = step;
    cfg.host_out = out; cfg.out_frame_stride = out_frame_stride; cfg.out_step = out_step;
    return offline_job(o, &cfg, nullptr, 1, 0);
}

// =====================================================================================
// simulator render + single-kernel entry points (host buffers)
// =====================================================================================
// CameraParams (x y z pan tilt roll, include/camera_engine.hpp:44-74) -> the rotation the renderer uses:
// rotationMatrix = Rz(roll) * Rx(tilt) * Ry(pan), camera_engine.cpp:36-61 (products individually rounded, as cv::Mat's)
static void poses_to_render(const double* poses, long n, RenderPose* hp) {
    for (long i = 0; i < n; ++i) {
        const double* p = poses + (size_t)i * 6;
        const double pan = p[3] * M_PI / 180.0, tilt = p[4] * M_PI / 180.0, roll = p[5] * M_PI / 180.0;
        const double ry[9] = {cos(pan), 0, sin(pan), 0, 1, 0, -sin(pan), 0, cos(pan)};
        const double rx[9] = {1, 0, 0, 0, cos(tilt), -sin(tilt), 0, sin(tilt), cos(tilt)};
        const double rz[9] = {cos(roll), -sin(roll), 0, sin(roll), cos(roll), 0, 0, 0, 1};
        double t[9];
        auto mm = [](const double* A, const double* B, double* C) {
            for (int i = 0; i < 3; ++i)
                for (int j = 0; j < 3; ++j) {
                    volatile double s = 0.0;
                    for (int k = 0; k < 3; ++k) { volatile double pr = A[i * 3 + k] * B[k * 3 + j]; s = s + pr; }
                    C[i * 3 + j] = s;
                }
        };
        mm(rz, rx, t);
        mm(t, ry, hp[i].R);
        hp[i].cam[0] = p[0]; hp[i].cam[1] = p[1]; hp[i].cam[2] = p[2];
    }
}


extern "C" vstab_status vstab_render_frames(int device, const uint8_t* d_texture, int tex_rows, int tex_cols,
                                            const double* poses, int n, int rows, int cols, double focal,
                                            uint8_t* d_out, size_t frame_stride, size_t step) {
    auto set_err = [&](const std::string& e) { g_err = e; };
    if (!d_texture || !poses || !d_out || n < 1) return VSTAB_ERR_INVALID_ARGUMENT;
    if (!device_ok(device, g_err)) return VSTAB_ERR_CUDA;
    std::vector<RenderPose> hp(n);
    poses_to_render(poses, n, hp.data());
    DevBuf dp;
    CK(dp.alloc(sizeof(RenderPose) * n));
    CK(cudaMemcpy(dp.p, hp.data(), sizeof(RenderPose) * n, cudaMemcpyHostToDevice));
    launch_render(d_texture, tex_rows, tex_cols, dp.as<RenderPose>(), n, cols, rows, focal, d_out, step, frame_stride, 0);
    CK(cudaGetLastError());
    CK(cudaDeviceSynchronize());
    return VSTAB_OK;
}
extern "C" vstab_status vstab_k_ingest(int device, const uint8_t* bgr, int rows, int cols, size_t step,
                                       int working_height, uint8_t* gray_out, uint64_t sums_out[3]) {
    auto set_err = [&](const std::string& e) { g_err = e; };
    if (!bgr || !gray_out || !sums_out) return VSTAB_ERR_INVALID_ARGUMENT;
    if (!device_ok(device, g_err)) return VSTAB_ERR_CUDA;
    Geometry g;
    vstab_status st = g.init(rows, cols, working_height, g_err);
    if (st != VSTAB_OK) return st;
    DevBuf frame, gray, sums;
    CK(frame.alloc(g.frame_bytes + 64));
    CK(gray.alloc(g.pd.frame_bytes));
    CK(sums.alloc(sizeof(unsigned long long) * 3));
    CK(cudaMemcpy2D(frame.p, g.pitch, bgr, step, (size_t)cols * 3, rows, cudaMemcpyHostToDevice));
    CK(cudaMemset(sums.p, 0, sizeof(unsigned long long) * 3));
    launch_ingest(g.plan, frame.as<uint8_t>(), g.pitch, g.frame_bytes, 1, gray.as<uint8_t>(), g.pd.frame_bytes,
                  sums.as<unsigned long long>(), 0);
    CK(cudaGetLastError());
    CK(cudaMemcpy(gray_out, gray.p, (size_t)g.ww * g.wh, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(sums_out, sums.p, sizeof(unsigned long long) * 3, cudaMemcpyDeviceToHost));
    return VSTAB_OK;
}

extern "C" vstab_status vstab_k_pyramid(int device, const uint8_t* gray, int rows, int cols,
                                        uint8_t* l1, uint8_t* l2, uint8_t* l3) {
    auto set_err = [&](const std::string& e) { g_err = e; };
    if (!gray || !l1 || !l2 || !l3) return VSTAB_ERR_INVALID_ARGUMENT;
    if (!device_ok(device, g_err)) return VSTAB_ERR_CUDA;
    PyrDesc pd = make_pyr_desc(cols, rows);
    DevBuf pyr;
    CK(pyr.alloc(pd.frame_bytes));
    CK(cudaMemcpy(pyr.p, gray, (size_t)rows * cols, cudaMemcpyHostToDevice));
    launch_pyramid(pd, pyr.as<uint8_t>(), 1, 0);
    CK(cudaGetLastError());
    uint8_t* outs[3] = {l1, l2, l3};
    for (int l = 1; l < kLkLevels; ++l)
        CK(cudaMemcpy(outs[l - 1], pyr.as<uint8_t>() + pd.off[l], (size_t)pd.w[l] * pd.h[l], cudaMemcpyDeviceToHost));
    return VSTAB_OK;
}

extern "C" vstab_status vstab_k_gftt(int device, const uint8_t* gray, int rows, int cols, int max_corners,
                                     double quality, int min_distance, float* pts_out, int* n_out, float* eig_out) {
    auto set_err = [&](const std::string& e) { g_err = e; };
    if (!gray || !pts_out || !n_out) return VSTAB_ERR_INVALID_ARGUMENT;
    if (!device_ok(device, g_err)) return VSTAB_ERR_CUDA;
    DevBuf img, mem, pts, cnt;
    GfttWorkspace ws{};
    size_t bytes = gftt_workspace_bytes(cols, rows, min_distance, 1, &ws);
    CK(img.alloc((size_t)rows * cols));
    CK(mem.alloc(bytes));
    CK(pts.alloc(sizeof(float2) * kMaxCorners));
    CK(cnt.alloc(sizeof(int)));
    gftt_bind_workspace(mem.p, &ws);
    CK(cudaMemcpy(img.p, gray, (size_t)rows * cols, cudaMemcpyHostToDevice));
    launch_gftt(img.as<uint8_t>(), 0, cols, rows, 1, quality, min_distance, max_corners, ws, pts.as<float2>(),
                cnt.as<int>(), ws.eig, 0);
    CK(cudaGetLastError());
    CK(cudaMemcpy(n_out, cnt.p, sizeof(int), cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(pts_out, pts.p, sizeof(float2) * (*n_out), cudaMemcpyDeviceToHost));
    if (eig_out) CK(cudaMemcpy(eig_out, ws.eig, sizeof(float) * rows * cols, cudaMemcpyDeviceToHost));
    return VSTAB_OK;
}

extern "C" vstab_status vstab_k_lk(int device, const uint8_t* prev, const uint8_t* next, int rows, int cols,
                                   const float* pts, int n, float* out_pts, uint8_t* status) {
    auto set_err = [&](const std::string& e) { g_err = e; };
    if (!prev || !next || !pts || !out_pts || !status || n < 0 || n > kMaxCorners) return VSTAB_ERR_INVALID_ARGUMENT;
    if (!device_ok(device, g_err)) return VSTAB_ERR_CUDA;
    PyrDesc pd = make_pyr_desc(cols, rows);
    DevBuf p0, p1, dp, dc, dout, dst;
    CK(p0.alloc(pd.frame_bytes)); CK(p1.alloc(pd.frame_bytes));
    CK(dp.alloc(sizeof(float2) * kMaxCorners)); CK(dc.alloc(sizeof(int)));
    CK(dout.alloc(sizeof(float2) * kMaxCorners)); CK(dst.alloc(kMaxCorners));
    CK(cudaMemcpy(p0.p, prev, (size_t)rows * cols, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(p1.p, next, (size_t)rows * cols, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dp.p, pts, sizeof(float2) * n, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dc.p, &n, sizeof(int), cudaMemcpyHostToDevice));
    launch_pyramid(pd, p0.as<uint8_t>(), 1, 0);
    launch_pyramid(pd, p1.as<uint8_t>(), 1, 0);
    launch_lk(p0.as<uint8_t>(), p1.as<uint8_t>(), pd.frame_bytes, pd.frame_bytes, pd, dp.as<float2>(), dc.as<int>(), 1,
              dout.as<float2>(), dst.as<uint8_t>(), 0);
    CK(cudaGetLastError());
    CK(cudaMemcpy(out_pts, dout.p, sizeof(float2) * n, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(status, dst.p, n, cudaMemcpyDeviceToHost));
    return VSTAB_OK;
}

extern "C" vstab_status vstab_k_fit(int device, const float* prev_pts, const float* next_pts, const uint8_t* status,
                                    int n, double thresh, int work_w, int work_h, double M_out[6], double T_out[9],
                                    int counts_out[2]) {
    auto set_err = [&](const std::string& e) { g_err = e; };
    if (!prev_pts || !next_pts || !status || !T_out || n < 0 || n > kMaxCorners) return VSTAB_ERR_INVALID_ARGUMENT;
    if (!device_ok(device, g_err)) return VSTAB_ERR_CUDA;
    DevBuf a, b, s, c, T, M, fc;
    CK(a.alloc(sizeof(float2) * kMaxCorners)); CK(b.alloc(sizeof(float2) * kMaxCorners)); CK(s.alloc(kMaxCorners));
    CK(c.alloc(sizeof(int))); CK(T.alloc(sizeof(double) * 9)); CK(M.alloc(sizeof(double) * 6)); CK(fc.alloc(sizeof(int) * 2));
    CK(cudaMemcpy(a.p, prev_pts, sizeof(float2) * n, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(b.p, next_pts, sizeof(float2) * n, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(s.p, status, n, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(c.p, &n, sizeof(int), cudaMemcpyHostToDevice));
    launch_fit(a.as<float2>(), b.as<float2>(), s.as<uint8_t>(), c.as<int>(), 1, thresh, work_w / 2.0, work_h / 2.0,
               T.as<double>(), M.as<double>(), fc.as<int>(), nullptr, 0, 0);
    CK(cudaGetLastError());
    CK(cudaMemcpy(T_out, T.p, sizeof(double) * 9, cudaMemcpyDeviceToHost));
    if (M_out) CK(cudaMemcpy(M_out, M.p, sizeof(double) * 6, cudaMemcpyDeviceToHost));
    if (counts_out) CK(cudaMemcpy(counts_out, fc.p, sizeof(int) * 2, cudaMemcpyDeviceToHost));
    return VSTAB_OK;
}

extern "C" vstab_status vstab_k_warp(int device, const uint8_t* bgr, int rows, int cols, size_t step, const double H[9],
                                     const uint8_t border[3], uint8_t* out, size_t out_step) {
    auto set_err = [&](const std::string& e) { g_err = e; };
    if (!bgr || !H || !border || !out) return VSTAB_ERR_INVALID_ARGUMENT;
    if (!device_ok(device, g_err)) return VSTAB_ERR_CUDA;
    const size_t pitch = align_up((size_t)cols * 3, 16);
    DevBuf src, dst, wp;
    CK(src.alloc(pitch * rows + 64)); CK(dst.alloc(pitch * rows + 64)); CK(wp.alloc(sizeof(WarpParams)));
    CK(cudaMemcpy2D(src.p, pitch, bgr, step, (size_t)cols * 3, rows, cudaMemcpyHostToDevice));
    WarpParams h{};
    for (int i = 0; i < 9; ++i) { h.Hs[i] = H[i]; h.Hw[i] = H[i]; }
    invert3(H, h.Minv);
    h.src_slot = 0;
    h.border[0] = border[0]; h.border[1] = border[1]; h.border[2] = border[2]; h.border[3] = 0;
    CK(cudaMemcpy(wp.p, &h, sizeof(h), cudaMemcpyHostToDevice));
    launch_warp(src.as<uint8_t>(), pitch, 0, 0, wp.as<WarpParams>(), 1, cols, rows, dst.as<uint8_t>(), pitch, 0, 0);
    CK(cudaGetLastError());
    CK(cudaMemcpy2D(out, out_step, dst.p, pitch, (size_t)cols * 3, rows, cudaMemcpyDeviceToHost));
    return VSTAB_OK;
}

// K15 alone.  The YUV frame is mirrored on the device byte for byte over its extent (padding and gaps included), so the
// kernels run on the caller's layout -- padded steps, planes apart, unaligned offsets -- and the caller sees exactly which
// bytes bgr_to_yuv writes.
extern "C" vstab_status vstab_k_yuv_to_bgr(int device, const uint8_t* yuv, const vstab_yuv_layout* layout, int rows, int cols,
                                           uint8_t* bgr, size_t step) {
    auto set_err = [&](const std::string& e) { g_err = e; };
    if (!yuv || !bgr || step < (size_t)cols * 3) { g_err = "null pointer or row step smaller than 3*cols"; return VSTAB_ERR_INVALID_ARGUMENT; }
    const size_t extent = yuv_extent(layout, rows, cols, g_err);
    if (!extent) return VSTAB_ERR_INVALID_ARGUMENT;
    if (!device_ok(device, g_err)) return VSTAB_ERR_CUDA;
    const size_t pitch = align_up((size_t)cols * 3, 16);
    DevBuf src, dst;
    CK(src.alloc(extent)); CK(dst.alloc(pitch * rows));
    CK(cudaMemcpy(src.p, yuv, extent, cudaMemcpyHostToDevice));
    launch_yuv420_to_bgr(src.as<uint8_t>(), yuv_planes_of(*layout), 0, 1, rows, cols, dst.as<uint8_t>(), pitch, 0, 0);
    CK(cudaGetLastError());
    CK(cudaMemcpy2D(bgr, step, dst.p, pitch, (size_t)cols * 3, rows, cudaMemcpyDeviceToHost));
    return VSTAB_OK;
}

extern "C" vstab_status vstab_k_bgr_to_yuv(int device, const uint8_t* bgr, int rows, int cols, size_t step, uint8_t* yuv,
                                           const vstab_yuv_layout* layout) {
    auto set_err = [&](const std::string& e) { g_err = e; };
    if (!yuv || !bgr || step < (size_t)cols * 3) { g_err = "null pointer or row step smaller than 3*cols"; return VSTAB_ERR_INVALID_ARGUMENT; }
    const size_t extent = yuv_extent(layout, rows, cols, g_err);
    if (!extent) return VSTAB_ERR_INVALID_ARGUMENT;
    if (!device_ok(device, g_err)) return VSTAB_ERR_CUDA;
    const size_t pitch = align_up((size_t)cols * 3, 16);
    DevBuf src, dst;
    CK(src.alloc(pitch * rows)); CK(dst.alloc(extent));
    CK(cudaMemcpy2D(src.p, pitch, bgr, step, (size_t)cols * 3, rows, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dst.p, yuv, extent, cudaMemcpyHostToDevice));
    launch_bgr_to_yuv420(src.as<uint8_t>(), pitch, 0, 1, rows, cols, dst.as<uint8_t>(), yuv_planes_of(*layout), 0, 0);
    CK(cudaGetLastError());
    CK(cudaMemcpy(yuv, dst.p, extent, cudaMemcpyDeviceToHost));
    return VSTAB_OK;
}

extern "C" vstab_status vstab_set_partial_lock_fix(vstab_t* s, int enable) {
    if (!s) return VSTAB_ERR_INVALID_ARGUMENT;
    if (s->partial_fix == (enable != 0)) return VSTAB_OK;
    s->partial_fix = enable != 0;
    s->epoch += 1;
    if (s->mode == VSTAB_TRANSLATION_LOCK || s->mode == VSTAB_ROTATION_LOCK) {
        // the lock starts at the next call, as after setStabilizationMode (:55-70)
        s->acc_valid = false; s->acc_to = -1; s->acc_call = -1;
        s->lock_call = s->n;
    }
    return VSTAB_OK;
}

extern "C" vstab_status vstab_set_trail(vstab_t* s, int enable) {
    if (!s) return VSTAB_ERR_INVALID_ARGUMENT;
    s->trail = enable != 0;
    s->epoch += 1;                       // an output prepared ahead without the trail is dropped
    return VSTAB_OK;
}

extern "C" vstab_status vstab_set_crop(vstab_t* s, double max_zoom, double release) {
    if (!s) return VSTAB_ERR_INVALID_ARGUMENT;
    if (!crop_params(max_zoom, release, &s->crop, s->err)) return VSTAB_ERR_INVALID_ARGUMENT;
    s->crop_reset = true;
    s->epoch += 1;                       // an output prepared ahead with the old crop is dropped
    return VSTAB_OK;
}

extern "C" double vstab_crop_zoom(const double H[9], int rows, int cols, double max_zoom) {
    if (!H || rows < 2 || cols < 2 || !(max_zoom >= 1.0 && max_zoom <= 4.0)) return -1.0;
    return crop_need(H, rows, cols, max_zoom);
}

extern "C" vstab_status vstab_k_copy_feathered(int device, const uint8_t* fg, const uint8_t* bg, int rows, int cols, size_t step,
                                               const double H[9], uint8_t* out, size_t out_step) {
    auto set_err = [&](const std::string& e) { g_err = e; };
    if (!fg || !bg || !H || !out || rows < 1 || cols < 1) return VSTAB_ERR_INVALID_ARGUMENT;
    if (!finite9(H)) { g_err = "Stabilizer: copyFeathered: Bad homography matrix H."; return VSTAB_ERR_INVALID_ARGUMENT; }
    if (!device_ok(device, g_err)) return VSTAB_ERR_CUDA;
    const size_t pitch = align_up((size_t)cols * 3, 16);
    const size_t fb = align_up(pitch * (size_t)rows, 256);
    DevBuf dfg, dbg, dout, wp, ws;
    CK(dfg.alloc(fb + 64)); CK(dbg.alloc(fb + 64)); CK(dout.alloc(fb + 64)); CK(wp.alloc(sizeof(WarpParams)));
    CK(ws.alloc(trail_workspace_bytes(cols, rows, fb)));
    CK(cudaMemcpy2D(dfg.p, pitch, fg, step, (size_t)cols * 3, rows, cudaMemcpyHostToDevice));
    CK(cudaMemcpy2D(dbg.p, pitch, bg, step, (size_t)cols * 3, rows, cudaMemcpyHostToDevice));
    WarpParams h{};
    for (int i = 0; i < 9; ++i) { h.Hs[i] = H[i]; h.Hw[i] = H[i]; }
    invert3(H, h.Minv);
    CK(cudaMemcpy(wp.p, &h, sizeof(h), cudaMemcpyHostToDevice));
    launch_trail(dfg.as<uint8_t>(), pitch, 0, 0, wp.as<WarpParams>(), 0, dbg.as<uint8_t>(), cols, rows, ws.p, dout.as<uint8_t>(), pitch, 0);
    CK(cudaGetLastError());
    CK(cudaMemcpy2D(out, out_step, dout.p, pitch, (size_t)cols * 3, rows, cudaMemcpyDeviceToHost));
    return VSTAB_OK;
}

// ---- ORB / SIFT registration path: single-kernel entry points (host buffers) ------------------
extern "C" vstab_status vstab_k_featprep(int device, const uint8_t* bgr, int rows, int cols, size_t step,
                                         int working_height, uint8_t* gray_out) {
    auto set_err = [&](const std::string& e) { g_err = e; };
    if (!bgr || !gray_out) return VSTAB_ERR_INVALID_ARGUMENT;
    if (!device_ok(device, g_err)) return VSTAB_ERR_CUDA;
    Geometry g;
    vstab_status st = g.init(rows, cols, working_height, g_err);
    if (st != VSTAB_OK) return st;
    DevBuf frame, ws, out;
    CK(frame.alloc(g.frame_bytes + 64));
    CK(ws.alloc(featprep_workspace_bytes(g.ww, g.wh)));
    CK(out.alloc((size_t)g.ww * g.wh));
    CK(g.nn_tables());
    CK(cudaMemcpy2D(frame.p, g.pitch, bgr, step, (size_t)cols * 3, rows, cudaMemcpyHostToDevice));
    launch_featprep(frame.as<uint8_t>(), g.pitch, g.nn_x.as<int>(), g.nn_y.as<int>(), g.ww, g.wh, ws.p, out.as<uint8_t>(), 0);
    CK(cudaGetLastError());
    CK(cudaMemcpy(gray_out, out.p, (size_t)g.ww * g.wh, cudaMemcpyDeviceToHost));
    return VSTAB_OK;
}

// vstab_k_orb / vstab_k_sift: one detector run on a host gray image.  `launch(plan, img, kps, desc, count)` enqueues it on
// the default stream; keypoints come out as {x, y, size, angle, response, octave} floats, descriptors `width` bytes each.
template <class Plan, class Launch>
static vstab_status k_detect(int device, Plan* (*create)(int, int, double, int, std::string*), void (*destroy)(Plan*),
                             const char* name, int width, const uint8_t* gray, int rows, int cols, double size_ratio,
                             float* kps_out, uint8_t* desc_out, int* n_out, int max_out, Launch&& launch) {
    if (!gray || !kps_out || !desc_out || !n_out || max_out < 1) return VSTAB_ERR_INVALID_ARGUMENT;
    if (!device_ok(device, g_err)) return VSTAB_ERR_CUDA;
    Plan* P = create(cols, rows, size_ratio, kOrbMaxKp, &g_err);
    if (!P) return VSTAB_ERR_CUDA;
    DevBuf img, kps, desc, cnt;
    vstab_status st = VSTAB_OK;
    auto fail = [&](const std::string& m) { g_err = m; st = VSTAB_ERR_CUDA; };
    if (img.alloc((size_t)rows * cols) != cudaSuccess || kps.alloc(sizeof(OrbKeypoint) * kOrbMaxKp) != cudaSuccess ||
        desc.alloc((size_t)width * kOrbMaxKp) != cudaSuccess || cnt.alloc(sizeof(int)) != cudaSuccess) fail("cudaMalloc failed");
    if (st == VSTAB_OK) {
        cudaMemcpy(img.p, gray, (size_t)rows * cols, cudaMemcpyHostToDevice);
        launch(P, img.as<uint8_t>(), kps.as<OrbKeypoint>(), desc.as<uint8_t>(), cnt.as<int>());
        int n = 0;
        if (cudaMemcpy(&n, cnt.p, sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess) fail(cudaGetErrorString(cudaGetLastError()));
        if (st == VSTAB_OK) {
            if (n > kOrbMaxKp) n = kOrbMaxKp;
            if (n > max_out) n = max_out;
            *n_out = n;
            std::vector<OrbKeypoint> h(n);
            cudaMemcpy(h.data(), kps.p, sizeof(OrbKeypoint) * n, cudaMemcpyDeviceToHost);
            cudaMemcpy(desc_out, desc.p, (size_t)width * n, cudaMemcpyDeviceToHost);
            for (int i = 0; i < n; ++i) {
                float* o = kps_out + (size_t)i * 6;
                o[0] = h[i].x; o[1] = h[i].y; o[2] = h[i].size; o[3] = h[i].angle; o[4] = h[i].response; o[5] = (float)h[i].octave;
            }
            if (cudaGetLastError() != cudaSuccess) fail(std::string("CUDA failure in ") + name);
        }
    }
    destroy(P);
    return st;
}

extern "C" vstab_status vstab_k_orb(int device, const uint8_t* gray, int rows, int cols, double size_ratio,
                                    int reference_order, float* kps_out, uint8_t* desc_out, int* n_out, int max_out) {
    return k_detect(device, orb_plan_create, orb_plan_destroy, "vstab_k_orb", 32, gray, rows, cols, size_ratio, kps_out, desc_out,
                    n_out, max_out, [&](OrbPlan* P, const uint8_t* img, OrbKeypoint* k, uint8_t* d, int* c) {
                        launch_orb(P, img, k, d, c, reference_order != 0, 0);
                    });
}

extern "C" vstab_status vstab_k_hamming(int device, const uint8_t* ref, int nref, const uint8_t* cur, int ncur, float ratio,
                                        int* best_idx, int* best_d, int* second_d, uint8_t* good) {
    auto set_err = [&](const std::string& e) { g_err = e; };
    if (!ref || !cur || !best_idx || !best_d || !second_d || !good || nref < 0 || ncur < 0 || nref > kOrbMaxKp || ncur > kOrbMaxKp)
        return VSTAB_ERR_INVALID_ARGUMENT;
    if (!device_ok(device, g_err)) return VSTAB_ERR_CUDA;
    DevBuf a, b, na, nb, bi, bd, sd, gd, ka, kb, rp, cp, stt, nm;
    CK(a.alloc(32 * kOrbMaxKp)); CK(b.alloc(32 * kOrbMaxKp)); CK(na.alloc(4)); CK(nb.alloc(4));
    CK(bi.alloc(4 * kOrbMaxKp)); CK(bd.alloc(4 * kOrbMaxKp)); CK(sd.alloc(4 * kOrbMaxKp)); CK(gd.alloc(kOrbMaxKp));
    CK(ka.alloc(sizeof(OrbKeypoint) * kOrbMaxKp)); CK(kb.alloc(sizeof(OrbKeypoint) * kOrbMaxKp));
    CK(rp.alloc(sizeof(float2) * kOrbMaxKp)); CK(cp.alloc(sizeof(float2) * kOrbMaxKp)); CK(stt.alloc(kOrbMaxKp)); CK(nm.alloc(4));
    CK(cudaMemset(ka.p, 0, sizeof(OrbKeypoint) * kOrbMaxKp)); CK(cudaMemset(kb.p, 0, sizeof(OrbKeypoint) * kOrbMaxKp));
    CK(cudaMemcpy(a.p, ref, (size_t)32 * nref, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(b.p, cur, (size_t)32 * ncur, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(na.p, &nref, 4, cudaMemcpyHostToDevice)); CK(cudaMemcpy(nb.p, &ncur, 4, cudaMemcpyHostToDevice));
    launch_hamming_match(a.as<uint8_t>(), na.as<int>(), ka.as<OrbKeypoint>(), b.as<uint8_t>(), nb.as<int>(), kb.as<OrbKeypoint>(),
                         kOrbMaxKp, ratio, bi.as<int>(), bd.as<int>(), sd.as<int>(), gd.as<uint8_t>(), rp.as<float2>(),
                         cp.as<float2>(), stt.as<uint8_t>(), nm.as<int>(), 0);
    CK(cudaGetLastError());
    CK(cudaMemcpy(best_idx, bi.p, 4 * (size_t)nref, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(best_d, bd.p, 4 * (size_t)nref, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(second_d, sd.p, 4 * (size_t)nref, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(good, gd.p, (size_t)nref, cudaMemcpyDeviceToHost));
    return VSTAB_OK;
}

extern "C" vstab_status vstab_k_l2match(int device, const uint8_t* ref, int nref, const uint8_t* cur, int ncur,
                                        int* best_idx, int* best_d2, uint8_t* good) {
    auto set_err = [&](const std::string& e) { g_err = e; };
    if (!ref || !cur || !best_idx || !best_d2 || !good || nref < 0 || ncur < 0 || nref > kOrbMaxKp || ncur > kOrbMaxKp)
        return VSTAB_ERR_INVALID_ARGUMENT;
    if (!device_ok(device, g_err)) return VSTAB_ERR_CUDA;
    DevBuf a, b, na, nb, bi, bd, gd, ka, kb, rp, cp, stt, nm, scr;
    CK(scr.alloc(l2_match_scratch_bytes(kOrbMaxKp, 1)));
    CK(a.alloc(128 * kOrbMaxKp)); CK(b.alloc(128 * kOrbMaxKp)); CK(na.alloc(4)); CK(nb.alloc(4));
    CK(bi.alloc(4 * kOrbMaxKp)); CK(bd.alloc(4 * kOrbMaxKp)); CK(gd.alloc(kOrbMaxKp));
    CK(ka.alloc(sizeof(OrbKeypoint) * kOrbMaxKp)); CK(kb.alloc(sizeof(OrbKeypoint) * kOrbMaxKp));
    CK(rp.alloc(sizeof(float2) * kOrbMaxKp)); CK(cp.alloc(sizeof(float2) * kOrbMaxKp)); CK(stt.alloc(kOrbMaxKp)); CK(nm.alloc(4));
    CK(cudaMemset(ka.p, 0, sizeof(OrbKeypoint) * kOrbMaxKp)); CK(cudaMemset(kb.p, 0, sizeof(OrbKeypoint) * kOrbMaxKp));
    CK(cudaMemcpy(a.p, ref, (size_t)128 * nref, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(b.p, cur, (size_t)128 * ncur, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(na.p, &nref, 4, cudaMemcpyHostToDevice)); CK(cudaMemcpy(nb.p, &ncur, 4, cudaMemcpyHostToDevice));
    if (!launch_l2_match(a.as<uint8_t>(), na.as<int>(), ka.as<OrbKeypoint>(), b.as<uint8_t>(), nb.as<int>(), kb.as<OrbKeypoint>(),
                         kOrbMaxKp, scr.p, bi.as<int>(), bd.as<int>(), gd.as<uint8_t>(), rp.as<float2>(), cp.as<float2>(),
                         stt.as<uint8_t>(), nm.as<int>(), 0)) { g_err = kL2MapErr; return VSTAB_ERR_CUDA; }
    CK(cudaGetLastError());
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpy(best_idx, bi.p, 4 * (size_t)nref, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(best_d2, bd.p, 4 * (size_t)nref, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(good, gd.p, (size_t)nref, cudaMemcpyDeviceToHost));
    return VSTAB_OK;
}

// The nearest-neighbour search of K12 for a batch of current sets against one reference set in ONE launch (frames stacked
// along the grid's z axis): cur is [nframes][max_rows][128], ncur[nframes]; results [nframes][nref].  `reps` > 1 repeats the
// launch and returns the average device time in *ms_out (CUDA events) for the tensor-pipe measurement.
extern "C" vstab_status vstab_k_l2match_batch(int device, const uint8_t* ref, int nref, const uint8_t* cur, const int* ncur,
                                              int nframes, int* best_idx, int* best_d2, int reps, float* ms_out) {
    auto set_err = [&](const std::string& e) { g_err = e; };
    if (!ref || !cur || !ncur || !best_idx || !best_d2 || nref < 0 || nref > kOrbMaxKp || nframes < 1 || nframes > 256) return VSTAB_ERR_INVALID_ARGUMENT;
    for (int f = 0; f < nframes; ++f) if (ncur[f] < 0 || ncur[f] > kOrbMaxKp) return VSTAB_ERR_INVALID_ARGUMENT;
    if (!device_ok(device, g_err)) return VSTAB_ERR_CUDA;
    DevBuf a, b, na, nb, bi, bd, scr;
    CK(a.alloc((size_t)128 * kOrbMaxKp)); CK(b.alloc((size_t)128 * kOrbMaxKp * nframes)); CK(na.alloc(4)); CK(nb.alloc(4 * (size_t)nframes));
    CK(bi.alloc(4 * (size_t)kOrbMaxKp * nframes)); CK(bd.alloc(4 * (size_t)kOrbMaxKp * nframes));
    CK(scr.alloc(l2_match_scratch_bytes(kOrbMaxKp, nframes)));
    CK(cudaMemset(a.p, 0, (size_t)128 * kOrbMaxKp)); CK(cudaMemset(b.p, 0, (size_t)128 * kOrbMaxKp * nframes));
    CK(cudaMemcpy(a.p, ref, (size_t)128 * nref, cudaMemcpyHostToDevice));
    size_t off = 0;
    for (int f = 0; f < nframes; ++f) {
        CK(cudaMemcpy(b.as<uint8_t>() + (size_t)f * kOrbMaxKp * 128, cur + off, (size_t)128 * ncur[f], cudaMemcpyHostToDevice));
        off += (size_t)128 * ncur[f];
    }
    CK(cudaMemcpy(na.p, &nref, 4, cudaMemcpyHostToDevice)); CK(cudaMemcpy(nb.p, ncur, 4 * (size_t)nframes, cudaMemcpyHostToDevice));
    if (!launch_l2_nn_batch(a.as<uint8_t>(), na.as<int>(), b.as<uint8_t>(), nb.as<int>(), kOrbMaxKp, nframes, scr.p, bi.as<int>(),
                            bd.as<int>(), 0)) { g_err = kL2MapErr; return VSTAB_ERR_CUDA; }                     // warm-up
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    const int R = reps > 0 ? reps : 1;
    CK(cudaEventRecord(e0, 0));
    for (int r = 0; r < R; ++r)              // the same descriptor arrays as the warm-up: their tensor maps are made again
        launch_l2_nn_batch(a.as<uint8_t>(), na.as<int>(), b.as<uint8_t>(), nb.as<int>(), kOrbMaxKp, nframes, scr.p, bi.as<int>(), bd.as<int>(), 0);
    CK(cudaEventRecord(e1, 0));
    CK(cudaDeviceSynchronize());
    CK(cudaGetLastError());
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    if (ms_out) *ms_out = ms / (float)R;
    for (int f = 0; f < nframes; ++f) {
        CK(cudaMemcpy(best_idx + (size_t)f * nref, bi.as<int>() + (size_t)f * kOrbMaxKp, 4 * (size_t)nref, cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(best_d2 + (size_t)f * nref, bd.as<int>() + (size_t)f * kOrbMaxKp, 4 * (size_t)nref, cudaMemcpyDeviceToHost));
    }
    return VSTAB_OK;
}

extern "C" vstab_status vstab_k_sift(int device, const uint8_t* gray, int rows, int cols, double size_ratio,
                                     float* kps_out, uint8_t* desc_out, int* n_out, int max_out) {
    return k_detect(device, sift_plan_create, sift_plan_destroy, "vstab_k_sift", 128, gray, rows, cols, size_ratio, kps_out, desc_out,
                    n_out, max_out, [](SiftPlan* P, const uint8_t* img, OrbKeypoint* k, uint8_t* d, int* c) {
                        launch_sift(P, img, k, d, c, 0);
                    });
}

// K11 with its stages read back (stage tests): `calls` runs of launch_sift on ONE plan and one non-blocking stream (the
// second call captures the CUDA graph, later calls replay it); everything returned is from the last call.
extern "C" vstab_status vstab_k_sift_stages(int device, const uint8_t* gray, int rows, int cols, double size_ratio, int calls,
                                            int* geom, float* pyr, size_t pyr_cap, uint64_t* cand, int cand_max,
                                            float* kps_pre, int kp_max, int counts[5], float* kps_out, uint8_t* desc_out,
                                            int* n_out, int max_out) {
    auto set_err = [&](const std::string& e) { g_err = e; };
    if (!gray || !geom || !counts || !kps_out || !desc_out || !n_out || rows < 1 || cols < 1 || calls < 1 || max_out < 1 ||
        (cand && cand_max < 0) || (kps_pre && kp_max < 0))
        return VSTAB_ERR_INVALID_ARGUMENT;
    if (!device_ok(device, g_err)) return VSTAB_ERR_CUDA;
    std::unique_ptr<SiftPlan, void (*)(SiftPlan*)> P(sift_plan_create(cols, rows, size_ratio, kOrbMaxKp, &g_err), sift_plan_destroy);
    if (!P) return VSTAB_ERR_CUDA;
    int w[kSiftMaxOctaves] = {}, h[kSiftMaxOctaves] = {};
    size_t off[kSiftMaxOctaves] = {};
    const int n_oct = sift_plan_geometry(P.get(), w, h, off);
    geom[0] = n_oct;
    for (int o = 0; o < kSiftMaxOctaves; ++o) {
        geom[1 + o] = w[o]; geom[1 + kSiftMaxOctaves + o] = h[o]; geom[1 + 2 * kSiftMaxOctaves + o] = (int)off[o];
    }
    if (pyr && pyr_cap < P->pyr_floats) {
        g_err = "vstab_k_sift_stages: the pyramid needs " + std::to_string(P->pyr_floats) + " floats";
        return VSTAB_ERR_INVALID_ARGUMENT;
    }
    DevBuf img, kps, desc, cnt;
    CK(img.alloc((size_t)rows * cols)); CK(kps.alloc(sizeof(OrbKeypoint) * kOrbMaxKp)); CK(desc.alloc((size_t)128 * kOrbMaxKp));
    CK(cnt.alloc(sizeof(int)));
    cudaStream_t st = nullptr;
    CK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    // the upload is ordered before the first launch on the same stream (a pageable cudaMemcpy on the legacy stream is not)
    cudaMemcpyAsync(img.p, gray, (size_t)rows * cols, cudaMemcpyHostToDevice, st);
    for (int c = 0; c < calls; ++c) launch_sift(P.get(), img.as<uint8_t>(), kps.as<OrbKeypoint>(), desc.as<uint8_t>(), cnt.as<int>(), st);
    const cudaError_t e = cudaStreamSynchronize(st);
    cudaStreamDestroy(st);
    CK(e);
    CK(cudaGetLastError());
    int hc[3] = {0, 0, 0}, n = 0;
    CK(cudaMemcpy(hc, P->counters, sizeof(hc), cudaMemcpyDeviceToHost));
    counts[0] = hc[0]; counts[1] = P->cand_cap; counts[2] = hc[1]; counts[3] = P->kp_cap; counts[4] = hc[2];
    if (pyr) CK(cudaMemcpy(pyr, P->pyr, sizeof(float) * P->pyr_floats, cudaMemcpyDeviceToHost));
    if (cand) CK(cudaMemcpy(cand, P->cand, 8 * (size_t)std::min(std::min(hc[0], P->cand_cap), cand_max), cudaMemcpyDeviceToHost));
    if (kps_pre) CK(cudaMemcpy(kps_pre, P->kps, sizeof(OrbKeypoint) * (size_t)std::min(std::min(hc[1], P->kp_cap), kp_max),
                               cudaMemcpyDeviceToHost));      // SiftKp has OrbKeypoint's layout: the octave word is an int
    CK(cudaMemcpy(&n, cnt.p, sizeof(int), cudaMemcpyDeviceToHost));
    n = std::min(std::min(n, kOrbMaxKp), max_out);
    *n_out = n;
    std::vector<OrbKeypoint> hk(n);
    CK(cudaMemcpy(hk.data(), kps.p, sizeof(OrbKeypoint) * n, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(desc_out, desc.p, (size_t)128 * n, cudaMemcpyDeviceToHost));
    for (int i = 0; i < n; ++i) {
        float* o = kps_out + (size_t)i * 6;
        o[0] = hk[i].x; o[1] = hk[i].y; o[2] = hk[i].size; o[3] = hk[i].angle; o[4] = hk[i].response; o[5] = (float)hk[i].octave;
    }
    return VSTAB_OK;
}

// K5's estimator instantiated for kOrbMaxKp pairs (the ORB / SIFT registration fit), on one pair set of up to 4096 pairs
extern "C" vstab_status vstab_k_fit_large(int device, const float* ref_pts, const float* cur_pts, const uint8_t* status, int n,
                                          double thresh, int work_w, int work_h, double M_out[6], double T_out[9],
                                          int counts_out[2]) {
    auto set_err = [&](const std::string& e) { g_err = e; };
    if (!ref_pts || !cur_pts || !status || !T_out || n < 0 || n > kOrbMaxKp) return VSTAB_ERR_INVALID_ARGUMENT;
    if (!device_ok(device, g_err)) return VSTAB_ERR_CUDA;
    DevBuf a, b, s, c, T, M, fc;
    CK(a.alloc(sizeof(float2) * kOrbMaxKp)); CK(b.alloc(sizeof(float2) * kOrbMaxKp)); CK(s.alloc(kOrbMaxKp));
    CK(c.alloc(sizeof(int))); CK(T.alloc(sizeof(double) * 9)); CK(M.alloc(sizeof(double) * 6)); CK(fc.alloc(sizeof(int) * 2));
    CK(cudaMemcpy(a.p, ref_pts, sizeof(float2) * n, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(b.p, cur_pts, sizeof(float2) * n, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(s.p, status, n, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(c.p, &n, sizeof(int), cudaMemcpyHostToDevice));
    launch_fit_large(a.as<float2>(), b.as<float2>(), s.as<uint8_t>(), c.as<int>(), thresh, work_w / 2.0, work_h / 2.0,
                     T.as<double>(), M.as<double>(), fc.as<int>(), 0);
    CK(cudaGetLastError());
    CK(cudaMemcpy(T_out, T.p, sizeof(double) * 9, cudaMemcpyDeviceToHost));
    if (M_out) CK(cudaMemcpy(M_out, M.p, sizeof(double) * 6, cudaMemcpyDeviceToHost));
    if (counts_out) CK(cudaMemcpy(counts_out, fc.p, sizeof(int) * 2, cudaMemcpyDeviceToHost));
    return VSTAB_OK;
}

// The DoG extrema pass of K11 alone, on a caller-made Gaussian pyramid of a rows x cols input (tests: values planted
// exactly at the contrast threshold).  pyr: the octaves of the plan's geometry (vstab_k_sift_stages' geom) one after the
// other without padding, each [6][h][w] float32.  cand / counts as vstab_k_sift_stages ({found, capacity}).
extern "C" vstab_status vstab_k_sift_extrema(int device, const float* pyr, size_t pyr_floats, int rows, int cols, uint64_t* cand,
                                             int cand_max, int counts[2]) {
    auto set_err = [&](const std::string& e) { g_err = e; };
    if (!pyr || !cand || !counts || rows < 1 || cols < 1 || cand_max < 0) return VSTAB_ERR_INVALID_ARGUMENT;
    if (!device_ok(device, g_err)) return VSTAB_ERR_CUDA;
    std::unique_ptr<SiftPlan, void (*)(SiftPlan*)> P(sift_plan_create(cols, rows, 0.0, kOrbMaxKp, &g_err), sift_plan_destroy);
    if (!P) return VSTAB_ERR_CUDA;
    int w[kSiftMaxOctaves] = {}, h[kSiftMaxOctaves] = {};
    size_t off[kSiftMaxOctaves] = {}, need = 0;
    const int n_oct = sift_plan_geometry(P.get(), w, h, off);
    for (int o = 0; o < n_oct; ++o) need += (size_t)6 * w[o] * h[o];
    if (pyr_floats != need) { g_err = "vstab_k_sift_extrema: the pyramid has " + std::to_string(need) + " floats"; return VSTAB_ERR_INVALID_ARGUMENT; }
    size_t src = 0;
    for (int o = 0; o < n_oct; ++o) {
        CK(cudaMemcpy(P->pyr + off[o], pyr + src, sizeof(float) * 6 * w[o] * h[o], cudaMemcpyHostToDevice));
        src += (size_t)6 * w[o] * h[o];
    }
    launch_sift_extrema(P.get(), 0);
    CK(cudaGetLastError());
    CK(cudaDeviceSynchronize());
    int n = 0;
    CK(cudaMemcpy(&n, P->counters, sizeof(int), cudaMemcpyDeviceToHost));
    counts[0] = n; counts[1] = P->cand_cap;
    CK(cudaMemcpy(cand, P->cand, 8 * (size_t)std::min(std::min(n, P->cand_cap), cand_max), cudaMemcpyDeviceToHost));
    return VSTAB_OK;
}
