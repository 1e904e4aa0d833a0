/*
 * vstab.h -- C ABI of the B200-native drop-in for the per-frame motion-estimation
 * and warp hot path of joao-gueifao-924/Video-Stabilization.
 *
 * Every entry point cites the reference interface it replaces
 * (paths relative to /root/reference).  There are no OpenCV, torch or C++ types
 * in any signature: plain pointers, sizes and PODs only.  The library has NO CPU
 * fallback: every compute entry point returns VSTAB_ERR_CUDA when no sm_100
 * device is usable.
 *
 * Images are 8-bit BGR, HWC, row-major with an explicit row step in bytes
 * (cv::Mat layout of include/stabilizer.hpp:67,86 and src/stabilizer.cpp:160).
 * Homographies are 3x3 row-major doubles (CV_64F, src/stabilizer.cpp:212).
 */
#ifndef VSTAB_H_
#define VSTAB_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VSTAB_ABI_VERSION 1

/* enum class StabilizationMode -- include/stabilizer.hpp:31-38 (same order/values) */
enum vstab_mode {
    VSTAB_ACCUMULATED_FULL_LOCK = 0,
    VSTAB_ORB_FULL_LOCK = 1,
    VSTAB_SIFT_FULL_LOCK = 2,
    VSTAB_TRANSLATION_LOCK = 3,
    VSTAB_ROTATION_LOCK = 4,
    VSTAB_GLOBAL_SMOOTHING = 5
};

/* Error behaviour of the reference (std::invalid_argument at src/stabilizer.cpp:40-49,
 * 99-114, 1438-1441) mapped to status codes; include/stabilizer.hpp re-raises them. */
typedef enum vstab_status {
    VSTAB_OK = 0,
    VSTAB_ERR_INVALID_ARGUMENT = 1, /* ctor / frame-size argument checks        */
    VSTAB_ERR_SIZE_CHANGED = 2,     /* "Frame size has changed" (:110-112)      */
    VSTAB_ERR_CUDA = 3,             /* no device / CUDA runtime failure          */
    VSTAB_ERR_UNSUPPORTED = 4,      /* mode not built yet (see DESIGN.md)        */
    VSTAB_ERR_STATE = 5,            /* call order the reference asserts against  */
    VSTAB_ERR_NCCL = 6              /* NCCL missing / a collective failed (sharded offline jobs only) */
} vstab_status;

/* struct HomographyParameters -- include/stabilizer.hpp:44-57 */
typedef struct vstab_hparams {
    double s;      /* isotropic scale          */
    double theta;  /* in-plane rotation [rad]  */
    double k;      /* anisotropy ratio k1      */
    double delta;  /* shear                    */
    double t[2];   /* translation              */
    double v[2];   /* horizon-line shift       */
} vstab_hparams;

typedef struct vstab vstab_t;               /* one Stabilizer instance == one CUDA stream */

/* ---- class Stabilizer ------------------------------------------------------------- */

/* Stabilizer::Stabilizer(pastFrames=15, futureFrames=15, workingHeight=360)
 * include/stabilizer.hpp:137, src/stabilizer.cpp:36-53 (same argument checks). */
vstab_status vstab_create(size_t past_frames, size_t future_frames, int working_height,
                          int device, vstab_t** out);
void vstab_destroy(vstab_t* s);

/* Stabilizer::setStabilizationMode -- include/stabilizer.hpp:188, src/stabilizer.cpp:55-96 */
vstab_status vstab_set_mode(vstab_t* s, int mode);
int vstab_get_mode(const vstab_t* s);

/* Stabilizer::totalFrameWindowSize -- include/stabilizer.hpp:196-198 */
size_t vstab_total_frame_window_size(const vstab_t* s);

/* cv::Mat Stabilizer::stabilizeFrame(const cv::Mat&) -- include/stabilizer.hpp:168,
 * src/stabilizer.cpp:1158-1325.  Host buffers; `bgr` may be reused by the caller as
 * soon as the call returns (the reference clones it, :160).  `out_bgr` receives the
 * stabilized presentation frame (call 0: a copy of the input, :1181). */
vstab_status vstab_stabilize_frame(vstab_t* s, const uint8_t* bgr, int rows, int cols,
                                   size_t step, uint8_t* out_bgr, size_t out_step);

/* Same call with device-resident input/output (both on the instance's device).
 * Asynchronous with respect to the host: work is enqueued on the instance stream;
 * call vstab_synchronize() before reading `d_out_bgr` from another stream. */
vstab_status vstab_stabilize_frame_device(vstab_t* s, const uint8_t* d_bgr, int rows, int cols,
                                          size_t step, uint8_t* d_out_bgr, size_t out_step);
vstab_status vstab_synchronize(vstab_t* s);

/* ---- YUV 4:2:0 frames (what video decoders produce and encoders take) ---------------------------------------------
 * NV12 (NVDEC's output: a Y plane and one interleaved U,V plane) and I420 (ffmpeg's yuv420p: Y, U, V planes), 8-bit,
 * BT.601 limited range.  The stabilizer stores and processes BGR either way: a YUV input frame is converted on the device
 * when it arrives, a BGR output frame is converted on the device before it leaves, each conversion exactly OpenCV's
 * (cvtColor COLOR_YUV2BGR_NV12 / _I420 and COLOR_BGR2YUV_I420; NV12 output = I420's chroma interleaved U,V).  So for every
 * call c:  out_yuv[c] == BGR2YUV_I420(stabilizeFrame(YUV2BGR(in_yuv))[c]) -- call 0 returns the converted copy of its
 * input converted back, not the caller's input bytes.  Only 1.5 bytes per pixel cross the host link instead of 3.
 * rows and cols must be even. */
typedef enum vstab_pixel_format { VSTAB_PIX_NV12 = 1, VSTAB_PIX_I420 = 2 } vstab_pixel_format;
/* plane k of a frame starts at base + offset[k] with rows step[k] bytes apart: k = 0 Y (rows x cols), NV12: k = 1 U,V
 * interleaved (rows/2 x cols bytes), k = 2 unused; I420: k = 1 U, k = 2 V (rows/2 x cols/2 each).  Covers ffmpeg's
 * data[] / linesize[] within one allocation and NVDEC's pitched surface with the chroma plane at pitch * rows. */
typedef struct vstab_yuv_layout {
    int format;                     /* vstab_pixel_format */
    size_t offset[3];
    size_t step[3];
} vstab_yuv_layout;
/* The tight rawvideo layout of a rows x cols frame (what `ffmpeg -f rawvideo -pix_fmt nv12|yuv420p` reads and writes)
 * into *out; returns the frame's size in bytes, or 0 for an unknown format, odd or non-positive sizes.  Host only. */
size_t vstab_yuv_layout_packed(int format, int rows, int cols, vstab_yuv_layout* out);
/* vstab_stabilize_frame / _device with YUV frames: `in` / `out` are frame base pointers, the layouts say where their planes
 * are (input and output formats are independent).  Same synchronicity as the BGR pair; BGR and YUV calls may be mixed on one
 * instance (the window holds BGR frames either way).  VSTAB_ERR_INVALID_ARGUMENT: NULL pointers or layouts, an unknown
 * format, odd rows or cols, a step below its plane's row bytes; the frame size checks are those of the BGR calls. */
vstab_status vstab_stabilize_frame_yuv(vstab_t* s, const uint8_t* in, const vstab_yuv_layout* in_layout, int rows, int cols,
                                       uint8_t* out, const vstab_yuv_layout* out_layout);
vstab_status vstab_stabilize_frame_yuv_device(vstab_t* s, const uint8_t* d_in, const vstab_yuv_layout* in_layout, int rows,
                                              int cols, uint8_t* d_out, const vstab_yuv_layout* out_layout);

/* static bool Stabilizer::decomposeHomography(H, params_out, rot_center)
 * include/stabilizer.hpp:227, src/stabilizer.cpp:1435-1533.
 * returns 1 (true) / 0 (false: degenerate, out untouched) / -1 (bad argument,
 * the reference throws std::invalid_argument).  Host-side double math, like the
 * reference; the device pipeline uses the same inline function (homography.cuh). */
int vstab_decompose_homography(const double H[9], double cx, double cy, vstab_hparams* out);

/* static cv::Mat Stabilizer::composeHomography(params, rot_center)
 * include/stabilizer.hpp:242, src/stabilizer.cpp:1535-1566 */
void vstab_compose_homography(const vstab_hparams* p, double cx, double cy, double H[9]);

/* The trail compositing branch of stabilizeFrame (src/stabilizer.cpp:1303-1307; `#if 0` in the reference, kept there for "GPU-
 * accelerated implementations", include/stabilizer.hpp:255-259): every output is copyFeathered(presentation frame,
 * trail background, H) and becomes the next trail background (zeros at the start, :128-130).  Off by default. */
vstab_status vstab_set_trail(vstab_t* s, int enable);

/* TRANSLATION_LOCK / ROTATION_LOCK as the reference's own formulas intend them (src/stabilizer.cpp:1246-1260:
 * R = getRotationMatrix2D(centre, theta(H_lock)), H_translation_lock = R * H_lock, H_rotation_lock = R^-1).  In the
 * reference calculateFullLockStabilization returns the identity in these two modes (:311-441), so both evaluate to the
 * identity ("@todo fix partial locking modes", include/stabilizer.hpp:23); that behaviour is the default here.  With
 * enable != 0 the two modes are fed with the ACCUMULATED_FULL_LOCK product (:317-338, anchor = the call after
 * setStabilizationMode): translation lock keeps the accumulated rotation and cancels the drift of the image centre,
 * rotation lock cancels only the accumulated rotation about the image centre.  Per-frame API only. */
vstab_status vstab_set_partial_lock_fix(vstab_t* s, int enable);

/* ---- auto-crop: zoom each output just enough to hide the border of its warp ---------------------------------------------
 * Beyond the reference (like vstab_set_trail): without it, wherever the warp reads outside the presentation frame the output
 * shows the border colour (half the frame's mean, src/stabilizer.cpp:1309).  Off by default (max_zoom == 1).
 * Notation: rows x cols the frame, c0 = ((cols-1)/2, (rows-1)/2), S = [0, cols-1] x [0, rows-1] the pixel centres, H_c the
 * H_stabilize_scaled of call c, Z(z) = [[z, 0, (1-z) c0x], [0, z, (1-z) c0y], [0, 0, 1]] the zoom by z about c0.
 *  1. need(H) (vstab_crop_zoom, f64, closed form): max_zoom if H is not finite or w = h20 x + h21 y + h22 <= 0 at a corner
 *     of S.  Else Q = H(S) is a convex quadrilateral; edge k runs Q[k] -> Q[k+1] (corners of S in the order (0,0),
 *     (cols-1,0), (cols-1,rows-1), (0,rows-1)), g = sign of Q's signed area (+1 when > 0, else -1).  Per edge (a, b):
 *     s0 = g cross(b-a, c0-a); s0 <= 0 (centre outside Q) -> max_zoom; per corner q of S, s1 = g cross(b-a, q-c0), and
 *     s1 < 0 bounds t <= s0 / -s1.  t* = min(1, every bound); need = clamp(1 / t*, 1, max_zoom).  need(I) == 1 exactly;
 *     a shift by dx needs ((cols-1)/2) / ((cols-1)/2 - |dx|).  No margin: the warp's 1/32-px source coordinates put a
 *     point within 1/64 px outside S on S, with zero weight on the taps outside it.
 *  2. zoom of call c (causal, so streaming and every offline split agree bit for bit):
 *     z_c = clamp(max over j in [max(0, c-R), c] of (n_j - (double)(c-j) * release), 1, max_zoom), n_j = need(H_j),
 *     R = ceil((max_zoom - 1) / release).  The zoom rises at once to what the current call needs and falls by at most
 *     `release` per call.  Streaming: calls before the call that enabled the crop count as n_j = 1.
 *  3. call c warps (or trails) with Hc = Z(z_c) * H_c, its inverse computed like H_c's.  Call 0 (H = I) stays the copy of
 *     its input.  Where z_c is capped at max_zoom a border can still show, in the usual colour.
 *  4. VSTAB_TAP_H_SCALED and vstab_offline_read_h report Hc; VSTAB_TAP_H_STABILIZE stays the working-resolution H.
 * Crop on: 1 < max_zoom <= 4, 0 < release (finite), R <= 4096; anything else (NaN included) is VSTAB_ERR_INVALID_ARGUMENT.
 * A switch drops an output prepared ahead, like vstab_set_trail; mode switches keep the history. */
vstab_status vstab_set_crop(vstab_t* s, double max_zoom, double release);
/* need(H) of rule 1 on the host: -1 for a NULL H, rows or cols < 2, or max_zoom outside [1, 4]. */
double vstab_crop_zoom(const double H[9], int rows, int cols, double max_zoom);
const char* vstab_last_error(const vstab_t* s);      /* message of the last non-OK status */
const char* vstab_status_string(vstab_status st);
int vstab_abi_version(void);

/* Pinned host memory for frame buffers (what cv::Mat's allocator is to the reference);
 * vstab_stabilize_frame() is fastest with buffers from here. */
void* vstab_host_alloc(size_t bytes);
void vstab_host_free(void* p);

/* ---- parity taps ------------------------------------------------------------------ */
/* Device->host dumps of the per-stage state after the most recent stabilize call, for
 * the parity tests (the reference has no equivalent; its state is private:
 * include/stabilizer.hpp:430-474). Each returns the element count written. */
typedef enum vstab_tap {
    VSTAB_TAP_GRAY = 0,        /* u8  working_h*working_w   current gray (src/stabilizer.cpp:1175) */
    VSTAB_TAP_PYR1 = 1,        /* u8  level-1 of the LK pyramid of the current gray               */
    VSTAB_TAP_PYR2 = 2,
    VSTAB_TAP_PYR3 = 3,
    VSTAB_TAP_PREV_PTS = 4,    /* f32 2*n   corners tracked in this call (prevPoints_, :1187)     */
    VSTAB_TAP_LK_PTS = 5,      /* f32 2*n   raw LK result for those corners                       */
    VSTAB_TAP_LK_STATUS = 6,   /* u8  n                                                           */
    VSTAB_TAP_NEW_PTS = 7,     /* f32 2*m   corners detected on the current gray (:1318)          */
    VSTAB_TAP_T = 8,           /* f64 9     transform pushed into the window (:1209)              */
    VSTAB_TAP_M = 9,           /* f64 6     similarity before scale kill (:224)                   */
    VSTAB_TAP_H_STABILIZE = 10,/* f64 9     H_stabilize (working-res, :1266-1288)                 */
    VSTAB_TAP_H_SCALED = 11,   /* f64 9     H_stabilize_scaled (:1291-1296)                       */
    VSTAB_TAP_BORDER = 12,     /* u8  3     border colour after saturate_cast (:1309)             */
    VSTAB_TAP_EIG = 13,        /* f32 working_h*working_w  min-eigenvalue map of the current gray (kept only with VSTAB_DEBUG_TAPS=1 in the environment) */
    VSTAB_TAP_INLIERS = 14,    /* i32 2     {n tracked, n RANSAC inliers}                         */
    VSTAB_TAP_CHANNEL_SUMS = 15,/* u64 3    per-channel byte sums of the presentation frame       */
    VSTAB_TAP_LOCK_H = 16,     /* f64 9     ORB registration: matrix returned by calculateFullLockStabilization (:784-787) */
    VSTAB_TAP_ORB_COUNTS = 17, /* i32 5     {keypoints current, reference, matches after ratio test, inliers, updated} */
    VSTAB_TAP_FEAT_GRAY = 18   /* u8  working_h*working_w  conditioned image of the presentation frame (:448-477) */
} vstab_tap;
long vstab_read_tap(vstab_t* s, int tap, void* dst, size_t dst_bytes);
int vstab_working_width(const vstab_t* s);
int vstab_working_height(const vstab_t* s);
long vstab_presentation_index(const vstab_t* s);    /* absolute index of the frame last output */

/* ---- offline (frame-sharded) mode ---------------------------------------------------
 * BASELINE.json north_star: a clip is sharded by contiguous frame ranges with a halo
 * frame; each GPU estimates its frame-pair transforms, the per-frame 3x3 are
 * all-gathered, then each GPU smooths and warps its own frames.  vstab_offline_run (below) is
 * that whole job behind one call; the functions here are its building blocks (device pointers,
 * caller-driven).  Index algebra: SURVEY.md Appendix C; results equal the
 * streaming calls above for every call index.  All pointers are DEVICE pointers. */
typedef struct vstab_offline vstab_offline_t;

vstab_status vstab_offline_create(size_t past_frames, size_t future_frames, int working_height,
                                  int rows, int cols, int max_batch, int device,
                                  vstab_offline_t** out);
void vstab_offline_destroy(vstab_offline_t* o);

/* Estimate T[f] (maps frame f-1 -> f, src/stabilizer.cpp:1187-1209) for the `n` frames
 * d_frames[0..n) whose absolute indices are first..first+n-1.  `d_halo` is frame first-1
 * (NULL when first == 0: T[0] is then identity and unused).  Writes 9 doubles per frame
 * to d_T[0..9n) and, when d_sums != NULL, the per-channel byte sums of each frame
 * (3 x u64 per frame: the cv::mean numerator of src/stabilizer.cpp:1309, a by-product of
 * the ingest pass) to d_sums[0..3n).  n <= max_batch. */
vstab_status vstab_offline_estimate(vstab_offline_t* o, const uint8_t* d_frames, size_t frame_stride,
                                    size_t step, int n, long first, const uint8_t* d_halo,
                                    double* d_T, unsigned long long* d_sums);

/* Produce the outputs of stabilizeFrame calls call_first..call_first+n-1 of a clip of
 * `n_total` frames given ALL transforms d_T_all[9*n_total] (T[0] ignored).  Call c
 * presents frame p = max(0, c - future); d_frames / d_sums are indexed by (p - frame_base).
 * mode: VSTAB_GLOBAL_SMOOTHING, or VSTAB_ACCUMULATED_FULL_LOCK with `lock_call` = the call
 * index at which setStabilizationMode was issued (>= future; earlier calls are smoothed). */
vstab_status vstab_offline_render(vstab_offline_t* o, const uint8_t* d_frames, size_t frame_stride,
                                  size_t step, long frame_base, int n, long call_first,
                                  const double* d_T_all, long n_total, int mode, long lock_call,
                                  const unsigned long long* d_sums,
                                  uint8_t* d_out, size_t out_frame_stride, size_t out_step);
/* Clip-wide preparation for a mode, given ALL transforms: for ACCUMULATED_FULL_LOCK the prefix
 * scan acc[k] = T[k]*...*T[anchor+1] (anchor = lock_call - future) over the 3x3 transforms
 * (src/stabilizer.cpp:317-338).  Must precede vstab_offline_render in that mode. */
vstab_status vstab_offline_prepare(vstab_offline_t* o, const double* d_T_all, long n_total, int mode,
                                   long lock_call);
/* Whole-clip stabilization with HOST buffers on one GPU (the reference's --file input,
 * src/main_utils.cpp:397-417 feeding stabilizeFrame at :465): `frames` holds n_total BGR frames
 * `frame_stride` bytes apart, `out` receives the outputs of stabilizeFrame calls 0..n_total-1.
 * This is vstab_offline_run (below) with a HOST source and host_out, as a world of one whatever
 * communicator the instance has joined: every mode is accepted, uploads, estimation, warping and
 * downloads are pipelined over chunks of max_batch frames, and device memory is bounded by the
 * chunk ring of the fused pass, not by the clip length; every frame crosses PCIe once per
 * direction (ORB / SIFT lock: uploaded twice, like the job's two passes).  Use pinned buffers
 * (vstab_host_alloc) for asynchronous copies.  Synchronous: returns when `out` is complete. */
vstab_status vstab_offline_run_host(vstab_offline_t* o, const uint8_t* frames, size_t frame_stride,
                                    size_t step, long n_total, int mode, long lock_call,
                                    uint8_t* out, size_t out_frame_stride, size_t out_step);
/* ORB_FULL_LOCK / SIFT_FULL_LOCK offline (SURVEY 8e): the owner of the anchor frame (the presentation frame
 * of the call at which the mode was set, src/stabilizer.cpp:520-589) captures the reference set and exports
 * it as one packed device buffer of vstab_offline_reference_bytes() bytes; the caller broadcasts it and
 * the other ranks import it.  Every rank then registers its own frames (independent units) into
 * d_reg[n][10] = {matrix[9], valid}; after the all-gather of those, vstab_offline_set_registrations +
 * vstab_offline_render apply the reference's "previously returned H" carry (:446) as a backward scan. */
size_t vstab_offline_reference_bytes(void);
vstab_status vstab_offline_reference_capture(vstab_offline_t* o, const uint8_t* d_frame, size_t step, int mode);
vstab_status vstab_offline_reference_export(vstab_offline_t* o, void* d_pack);
vstab_status vstab_offline_reference_import(vstab_offline_t* o, const void* d_pack, int mode);
vstab_status vstab_offline_register(vstab_offline_t* o, const uint8_t* d_frames, size_t frame_stride, size_t step,
                                    int n, double* d_reg);
vstab_status vstab_offline_set_registrations(vstab_offline_t* o, const double* d_reg_all, long n_total);
vstab_status vstab_offline_synchronize(vstab_offline_t* o);
const char* vstab_offline_last_error(const vstab_offline_t* o);   /* message of the last non-OK status of an offline instance */
/* per-stage device time (CUDA events on the instance stream) accumulated since the last call:
 * ms[8]/counts[8] = ingest, pyramid, gftt, lk, fit, smooth, warp, acc-scan */
void vstab_offline_set_timing(vstab_offline_t* o, int enable);
vstab_status vstab_offline_stage_times(vstab_offline_t* o, float* ms, int* counts);
/* number of this library's kernels launched by the process so far */
long long vstab_launch_count(void);
/* Measurement aid for bench.py's e2e leg: what the host link gives `device` with both directions busy.  Copies `bytes` of
 * pinned host memory host -> device (from host_in) and device -> host (into host_out) on two streams, in pieces of
 * chunk_bytes, `passes` times, no kernels; *seconds = wall time of the whole exchange. */
vstab_status vstab_debug_link_probe(int device, const void* host_in, void* host_out, size_t bytes, size_t chunk_bytes,
                                    int passes, double* seconds);
/* VSTAB_GUARD=1 in the environment puts every device buffer of the library between two 4 KB guard bands; when a buffer is
 * released the bands are read back.  Bytes found overwritten so far (out-of-bounds writes) / buffers allocated with bands. */
long long vstab_debug_guard_violations(void);
long long vstab_debug_guard_buffers(void);
/* device-side H_stabilize_scaled of the last render (9 doubles per call) for parity tests */
long vstab_offline_read_h(vstab_offline_t* o, double* dst, size_t n_calls);
/* cudaStream_t of the instance, as an integer handle, so callers can order NCCL work after it */
uintptr_t vstab_offline_stream(vstab_offline_t* o);

/* ---- sharded offline job: the whole multi-GPU path behind one call (SURVEY 8e, BASELINE config 5) ------------
 * One process per GPU.  Every rank creates a vstab_offline_t on its device, the ranks join one NCCL communicator
 * (rank 0 makes the id, the host program ships its 128 bytes to the others any way it likes), and every rank calls
 * vstab_offline_run with the same n_total / mode / lock_call:
 *   pass 1   rank r estimates T[f] for its contiguous range [first, last) (+ the halo frame first-1), chunk by chunk:
 *            a bounded number of frames is resident at any time (max_batch + 1; the fused pass below: its ring) -- the
 *            reference bounds memory the same way with its past+1+future window, stabilizer.cpp:160-167;
 *   exchange ONE ncclAllGather of 72 bytes per frame (ORB / SIFT lock: + one ncclBroadcast of the packed reference set
 *            and one all-gather of 80 bytes per frame {H, valid});
 *   pass 2   global prefix / window average for the calls whose presentation frame the rank owns, warp, sink.
 * Frames come from host memory (this rank's shard), from device memory, or from the simulator (K13 renders each
 * chunk on the device from `poses`: nothing of the clip is ever stored).  GLOBAL_SMOOTHING from a staged source (host,
 * simulator) runs the two passes as ONE: the window of call c reads T[c-P-F+1 .. c-1] only, so every call whose
 * window lies inside the rank's own transforms is warped right behind the estimation, out of a ring of the last
 * ceil((F-1)/max_batch) + 3 chunks (source, estimation and warp on three streams) -- a frame is uploaded / rendered
 * once; only the first P-1 and last F-1 calls of a rank in a world > 1 wait for the exchange and fetch their frames
 * again.  In a world of one the fused pass covers every LK-path mode (ACCUMULATED_FULL_LOCK rescans the prefix of the
 * transforms estimated so far before each warp step).  The other cases need the global prefix / the broadcast
 * reference and fetch every frame in both passes.  Outputs for host_out leave on a download stream of their own.
 * Outputs go to host memory and / or are reduced to one 64-bit checksum per call (see vstab_frame_checksum).  With no communicator the
 * instance is a world of one.  Replaces the reference's --file / --simulator loop around stabilizeFrame
 * (src/main_utils.cpp:397-417, 459-493) for clips that are sharded over GPUs. */
typedef struct vstab_nccl_id { char bytes[128]; } vstab_nccl_id;
vstab_status vstab_nccl_get_unique_id(vstab_nccl_id* out);                 /* rank 0 */
vstab_status vstab_offline_comm_init(vstab_offline_t* o, const vstab_nccl_id* id, int rank, int world);
/* frame range [first, last) and call range [call_first, call_last) of `rank` (balanced contiguous split; the owner of
 * frame 0 also produces the `future` warm-up calls; the last `future` frames are never presented, SURVEY B.5) */
typedef struct vstab_shard_plan { long first, last, call_first, call_last; } vstab_shard_plan;
vstab_status vstab_offline_plan(long n_total, int world, int rank, size_t future_frames, vstab_shard_plan* out);
/* the fused GLOBAL_SMOOTHING pass of a rank (staged sources): chunk k = frames [first + k*max_batch, ...) sits in ring slot
 * k % ring_chunks; the calls [fused_first, fused_last) are warped right behind the estimation (after chunk k: every call
 * c <= last frame of chunk k + 1), the calls [call_first, fused_first) and [fused_last, call_last) -- windows that reach
 * into a neighbour's shard -- after the all-gather.  The window of call c reads T[max(1, c-P-F+1) .. c-1]. */
typedef struct vstab_fused_plan { long ring_chunks, fused_first, fused_last; } vstab_fused_plan;
vstab_status vstab_offline_fused_plan(long n_total, int world, int rank, size_t past_frames, size_t future_frames,
                                      int max_batch, vstab_fused_plan* out);

typedef enum vstab_frame_source { VSTAB_SRC_HOST = 0, VSTAB_SRC_SIMULATOR = 1, VSTAB_SRC_DEVICE = 2 } vstab_frame_source;
typedef struct vstab_offline_cfg {
    long n_total;                   /* frames of the whole clip                                                  */
    int mode;                       /* vstab_mode; lock modes: lock_call = call index of setStabilizationMode      */
    long lock_call;
    int source;                     /* vstab_frame_source                                                          */
    /* VSTAB_SRC_HOST: this rank's frames [first, last) (pinned memory recommended) and frame first-1 (NULL on rank 0).
     * VSTAB_SRC_DEVICE: the same two pointers are DEVICE pointers (the shard is resident in HBM: no staging copies) */
    const uint8_t* host_frames; size_t frame_stride, step;
    const uint8_t* host_halo;
    /* VSTAB_SRC_SIMULATOR: device-resident BGR texture and the host array poses[n_total][6] = x y z pan tilt roll   */
    const uint8_t* d_texture; int tex_rows, tex_cols; const double* poses; double focal;
    /* sinks (each may be NULL): outputs of this rank's calls in call order, their checksums, all transforms         */
    uint8_t* host_out; size_t out_frame_stride, out_step;
    uint8_t* d_out;                 /* device sink with the same strides (instead of host_out)                     */
    uint64_t* checksums;            /* [call_last - call_first]                                                    */
    double* T_all;                  /* [n_total][9] host copy of the gathered transforms                           */
} vstab_offline_cfg;
typedef struct vstab_offline_report {   /* device time per phase on this rank, milliseconds (CUDA events)         */
    float source_ms, estimate_ms, exchange_ms, render_ms, total_ms;
    long frames, calls;
} vstab_offline_report;
vstab_status vstab_offline_run(vstab_offline_t* o, const vstab_offline_cfg* cfg, vstab_offline_report* report /* or NULL */);
/* YUV 4:2:0 frames for vstab_offline_run_host and vstab_offline_run (see vstab_yuv_layout above; NULL = BGR, the default):
 * `in` describes every source frame (HOST and DEVICE sources; the simulator source ignores it), `out` every output frame
 * (`out` / `host_out` / `d_out`).  While a layout is set the corresponding `step` / `out_step` arguments are ignored; frame
 * strides still apply and must cover the layout's planes.  Frames are converted on the device when they arrive and before
 * they leave; the clip is processed as BGR, so per-call checksums are those of the BGR outputs.  The device-pointer
 * building blocks (estimate, render, register, reference_capture) take BGR only.  VSTAB_ERR_INVALID_ARGUMENT for a
 * layout that does not fit the instance's frame size. */
vstab_status vstab_offline_set_yuv(vstab_offline_t* o, const vstab_yuv_layout* in, const vstab_yuv_layout* out);
/* Auto-crop (vstab_set_crop above, same parameters and semantics) for vstab_offline_render, _run_host and _run.  Every
 * render recomputes the matrices of the R calls before its first one, so the outputs equal the streaming calls' whatever
 * the batches or shards.  So with the crop on, the d_T_all of vstab_offline_render must hold T[max(1, call_first-R-P-F+1) ..],
 * and in vstab_offline_run's fused GLOBAL_SMOOTHING pass a call's matrices read like a window of past P + R (the fused plan
 * of past_frames + R: on ranks > 0 the first P + R - 1 calls wait for the exchange). */
vstab_status vstab_offline_set_crop(vstab_offline_t* o, double max_zoom, double release);
/* the checksum the warp kernel accumulates, of a host frame (tests) */
uint64_t vstab_frame_checksum(const uint8_t* bgr, int rows, int cols, size_t step);

/* ---- simulator frame source (CameraEngine::renderFrame, src/camera_engine.cpp:158-172) --
 * Renders `n` frames on the device from a device-resident BGR texture; poses are
 * (x, y, z, pan, tilt, roll) doubles per frame (CameraParams, include/camera_engine.hpp:44-74),
 * host pointer.  Used to feed synthetic clips without PCIe traffic. */
vstab_status vstab_render_frames(int device, const uint8_t* d_texture, int tex_rows, int tex_cols,
                                 const double* poses, int n, int rows, int cols, double focal,
                                 uint8_t* d_out, size_t frame_stride, size_t step);

/* ---- single-kernel entry points (host buffers; used by the kernel parity tests) ------ */
vstab_status vstab_k_ingest(int device, const uint8_t* bgr, int rows, int cols, size_t step,
                            int working_height, uint8_t* gray_out, uint64_t sums_out[3]);
vstab_status vstab_k_pyramid(int device, const uint8_t* gray, int rows, int cols,
                             uint8_t* l1, uint8_t* l2, uint8_t* l3);
vstab_status vstab_k_gftt(int device, const uint8_t* gray, int rows, int cols, int max_corners,
                          double quality, int min_distance, float* pts_out, int* n_out,
                          float* eig_out /* may be NULL */);
vstab_status vstab_k_lk(int device, const uint8_t* prev, const uint8_t* next, int rows, int cols,
                        const float* pts, int n, float* out_pts, uint8_t* status);
vstab_status vstab_k_fit(int device, const float* prev_pts, const float* next_pts,
                         const uint8_t* status, int n, double thresh, int work_w, int work_h,
                         double M_out[6], double T_out[9], int counts_out[2]);
/* the same estimator for up to 4096 pairs (the ORB / SIFT registration fit, one CTA on one pair set) */
vstab_status vstab_k_fit_large(int device, const float* ref_pts, const float* cur_pts,
                               const uint8_t* status, int n, double thresh, int work_w, int work_h,
                               double M_out[6], double T_out[9], int counts_out[2]);
vstab_status vstab_k_warp(int device, const uint8_t* bgr, int rows, int cols, size_t step,
                          const double H[9], const uint8_t border[3], uint8_t* out, size_t out_step);
/* Stabilizer::copyFeathered(foreground, background, H) (src/stabilizer.cpp:1051-1155): warp + feathered alpha blend over a
 * darkened, blurred gray background; both images rows x cols BGR with the same step. */
vstab_status vstab_k_copy_feathered(int device, const uint8_t* fg, const uint8_t* bg, int rows, int cols, size_t step,
                                    const double H[9], uint8_t* out, size_t out_step);
/* K15 alone: cvtColor(YUV2BGR_NV12 / _I420) and cvtColor(BGR2YUV_I420) (+ NV12 interleave) of one frame.  The YUV side is a
 * frame base pointer and its layout; bgr_to_yuv writes only the bytes of the layout's planes. */
vstab_status vstab_k_yuv_to_bgr(int device, const uint8_t* yuv, const vstab_yuv_layout* layout, int rows, int cols,
                                uint8_t* bgr, size_t step);
vstab_status vstab_k_bgr_to_yuv(int device, const uint8_t* bgr, int rows, int cols, size_t step, uint8_t* yuv,
                                const vstab_yuv_layout* layout);

/* ORB / SIFT registration path (src/stabilizer.cpp:448-477 preprocessing, :483-491 + :605-606 ORB
 * detectAndCompute, :647-673 Hamming 2-NN + ratio test).  kps_out: 6 floats per keypoint
 * {x, y, size, angle, response, octave}, level-major then row-major -- or, with reference_order,
 * in the exact order cv::ORB returns them (retainBest's nth_element permutation); desc_out: 32 bytes each. */
vstab_status vstab_k_featprep(int device, const uint8_t* bgr, int rows, int cols, size_t step,
                              int working_height, uint8_t* gray_out);
vstab_status vstab_k_orb(int device, const uint8_t* gray, int rows, int cols, double size_ratio,
                         int reference_order, float* kps_out, uint8_t* desc_out, int* n_out, int max_out);
vstab_status vstab_k_hamming(int device, const uint8_t* ref, int nref, const uint8_t* cur, int ncur,
                             float ratio, int* best_idx, int* best_d, int* second_d, uint8_t* good);

/* SIFT(2500, 3, 0.04, 5, 1.2).detectAndCompute (src/stabilizer.cpp:496-506, :614-615): kps_out 6 floats per
 * keypoint {x, y, size, angle, response, packed octave (cv::KeyPoint::octave)}, sorted by (x, y); desc_out
 * 128 bytes each (OpenCV stores the same integers as float). */
vstab_status vstab_k_sift(int device, const uint8_t* gray, int rows, int cols, double size_ratio,
                          float* kps_out, uint8_t* desc_out, int* n_out, int max_out);
/* vstab_k_sift with its stages read back (tests): `calls` runs on one plan (the second captures the CUDA graph, later
 * ones replay it), everything returned from the last.  geom[1 + 3 * 12]: octave count n, then w[12], h[12] of the
 * octaves (base image = 2x the input) and off[12].  pyr (may be NULL, else >= pyr_cap floats): the 6 Gaussians of
 * every octave, octave o as [6][h][w] float32 from pyr + off[o].  cand (may be NULL): the DoG extrema as
 * octave << 56 | layer << 48 | row << 24 | col, min(count, cap, cand_max) of them.  kps_pre (may be NULL): the refined,
 * oriented keypoints before duplicate removal and selection, {x, y, size, angle, response: float, octave: int32},
 * min(count, cap, kp_max) of them.  counts: {candidates found, candidate capacity, keypoints found, keypoint
 * capacity, keypoints selected}; a count above its capacity means entries were dropped (the selected keypoints
 * beyond max_out, 4096 at most, are dropped too: retainBest keeps every tie of its threshold).  kps_out / desc_out /
 * n_out as vstab_k_sift. */
vstab_status vstab_k_sift_stages(int device, const uint8_t* gray, int rows, int cols, double size_ratio, int calls,
                                 int* geom, float* pyr, size_t pyr_cap, uint64_t* cand, int cand_max,
                                 float* kps_pre, int kp_max, int counts[5], float* kps_out, uint8_t* desc_out,
                                 int* n_out, int max_out);
/* The DoG extrema pass of vstab_k_sift alone on a caller-made Gaussian pyramid for a rows x cols input (tests): pyr
 * holds the octaves of vstab_k_sift_stages' geometry one after the other without padding, each [6][h][w] float32,
 * pyr_floats in all; cand and counts ({found, capacity}) as vstab_k_sift_stages. */
vstab_status vstab_k_sift_extrema(int device, const float* pyr, size_t pyr_floats, int rows, int cols, uint64_t* cand,
                                  int cand_max, int counts[2]);
/* Exact L2 1-NN of SIFT descriptors (u8 [n][128]) on the tensor cores + the reference's distance filter
 * d <= max(0.5 * mean(d), 0.02) (src/stabilizer.cpp:675-697).  best_d2: exact squared distances. */
vstab_status vstab_k_l2match(int device, const uint8_t* ref, int nref, const uint8_t* cur, int ncur,
                             int* best_idx, int* best_d2, uint8_t* good);
/* The same nearest-neighbour search for `nframes` current sets (concatenated rows, ncur[f] rows each) against one reference
 * set in ONE launch; results [nframes][nref]; *ms_out (may be NULL) = device time of one launch averaged over `reps`. */
vstab_status vstab_k_l2match_batch(int device, const uint8_t* ref, int nref, const uint8_t* cur, const int* ncur, int nframes,
                                   int* best_idx, int* best_d2, int reps, float* ms_out);

#ifdef __cplusplus
}
#endif
#endif /* VSTAB_H_ */
