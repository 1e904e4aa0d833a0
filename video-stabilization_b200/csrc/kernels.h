// Host-callable launch wrappers of the hot-path kernels (all asynchronous on `st`).
// Layout conventions (device memory):
//   * BGR frames: u8 HWC, `pitch` bytes per row (multiple of 16), frames `frame_stride` apart.
//   * gray pyramid of a frame: one block of PyrDesc::frame_bytes, level l at off[l], tight rows.
//   * corners / LK points: float2 [frame][kMaxCorners]; counts int [frame].
//   * transforms: double [frame][9] row-major.
#pragma once
#include <mutex>
#include <string>
#include <vector>
#include "common.cuh"

namespace vstabk {

// number of kernels of this library launched so far (bench.py reports the delta per timed region)
void count_launch(int n);
long long launch_count();

// Function attributes (opt-in dynamic shared memory) and the SM count belong to a DEVICE, the C ABI takes a device per
// instance, and instances may live on several host threads: one-time setup is keyed by the current device and serialised.
struct PerDeviceOnce {
    std::mutex mu;
    unsigned long long done = 0;            // bit d: setup ran on device d
    template <class F>
    void run(F&& setup) {
        int dev = 0;
        cudaGetDevice(&dev);
        const unsigned long long bit = 1ull << (dev & 63);
        std::lock_guard<std::mutex> lock(mu);
        if (!(done & bit)) { setup(); done |= bit; }
    }
};
int device_sm_count();                      // of the current device (cached per device)

// ---------------------------------------------------------------- K1 ingest
struct IngestPlan {
    int src_w, src_h, dst_w, dst_h;
    int mode;              // 0 = copy (scale 1), 1 = exact 2x2 box (INTER_AREA), 2 = Q11 bilinear
    int rows_per_band;     // dst rows handled by one CTA
    int nbands;
    const int4* xtab;      // per dst x: {s0, s1, c0, c1}   (mode 2; also filled for 0/1)
    const int4* ytab;      // per dst y
};
void build_ingest_tables(int src, int dst, int mode, int4* host_tab);   // host helper
void launch_ingest(const IngestPlan& plan, const uint8_t* frames, size_t pitch, size_t frame_stride,
                   int nframes, uint8_t* gray, size_t gray_frame_stride,
                   unsigned long long* sums /* [nframes][3], pre-zeroed */, cudaStream_t st);

// ---------------------------------------------------------------- K2 pyramid
PyrDesc make_pyr_desc(int w, int h);
void launch_pyramid(const PyrDesc& d, uint8_t* pyr, int nframes, cudaStream_t st);

// ---------------------------------------------------------------- K3 GFTT
struct GfttWorkspace {
    float* eig;                    // [w*h]  one frame, written only when a parity tap asks for it
    unsigned int* maxbits;         // [nframes]
    unsigned long long* keys;      // [nframes][cap]
    unsigned long long* keys_alt;  // [nframes][cap]   (sort double buffer)
    int* seg_begin;                // [nframes]  = f*cap
    int* seg_end;                  // [nframes]  = f*cap + count (atomic counter)
    unsigned short* grid;          // [nframes][ncells*4] global fallback when the grid does not fit in smem
    void* cub_temp;
    size_t cub_temp_bytes;
    int cap;                       // candidate capacity per frame
    int ncells, grid_w, grid_h, cell;
    int grid_in_smem;
    int max_frames;
    int idx_bits;                  // candidate key = min-eigenvalue bits << idx_bits | pixel index
    int counters_ready;            // host flag: maxbits / seg_end were left reset by the fused kernel
};
size_t gftt_workspace_bytes(int w, int h, int min_distance, int max_frames, GfttWorkspace* layout);
void gftt_bind_workspace(void* base, GfttWorkspace* ws);     // base: cudaMalloc'ed block
void launch_gftt(const uint8_t* gray, size_t gray_frame_stride, int w, int h, int nframes,
                 double quality, int min_distance, int max_corners, GfttWorkspace& ws,
                 float2* pts, int* counts, float* eig_out /* [nframes][w*h] or null */, cudaStream_t st);

// ---------------------------------------------------------------- K4 sparse pyramidal LK
void launch_lk(const uint8_t* prev_pyr, const uint8_t* next_pyr, size_t prev_stride, size_t next_stride,
               const PyrDesc& d, const float2* pts, const int* counts, int nframes,
               float2* out_pts, uint8_t* status, cudaStream_t st);

// ---------------------------------------------------------------- K5 RANSAC similarity + LS + scale kill
void launch_fit(const float2* prev_pts, const float2* next_pts, const uint8_t* status,
                const int* counts, int nframes, double thresh, double cx, double cy,
                double* T /* [nframes][9] */, double* M /* [nframes][6] or null */,
                int* fit_counts /* [nframes][2] or null */, const long* frame_ids /* or null */,
                long frame_id0, cudaStream_t st);
// same estimator for up to kOrbMaxKp point pairs of ONE pair set (ORB / SIFT registration, thr 5.0, :734-736)
void launch_fit_large(const float2* ref_pts, const float2* cur_pts, const uint8_t* status, const int* count,
                      double thresh, double cx, double cy, double* T, double* M, int* fit_counts, cudaStream_t st);

// ---------------------------------------------------------------- K6 window smoothing / lock, warp params
struct WarpParams {          // consumed by K7
    double Minv[9];          // inverse of H_stabilize_scaled (dst -> src)
    double Hs[9];            // H_stabilize_scaled (tap)
    double Hw[9];            // H_stabilize at working resolution (tap)
    int src_slot;            // which source frame (index into the frame array / ring)
    unsigned char border[4]; // saturate_cast<uchar>(0.5*mean) per channel
};
struct SmoothArgs {
    const double* T;             // transforms by absolute frame index (T[k] maps k-1 -> k)
    long t_mod;                  // T index = abs % t_mod
    int P, F;                    // past / future window
    int mode;                    // vstab_mode
    long lock_call;              // call index at which the lock mode was set (ACCUMULATED)
    const double* acc;           // optional precomputed accumulated products by abs frame idx (offline), mod acc_mod
    long acc_mod;
    const double* lock_h;        // ORB / SIFT registration matrix (9 doubles, device) or null
    const double* reg;           // offline ORB / SIFT: per frame {H[9], valid} by absolute frame index, or null
    long reg_lo;                 // first frame a call after lock_call can present (lower end of the carry scan)
    double scale;                // workingHeight / rows
    const unsigned long long* sums;   // [slot][3] channel sums by frame slot; null: border left 0 (matrices only)
    long sums_mod;               // slot = abs frame % sums_mod   (ring) or abs - frame_base (offline: see frame_base)
    long frame_base;             // offline: slot = abs - frame_base; streaming: 0 with modulo
    double npix;                 // rows*cols
    int partial_fix;             // TRANSLATION_/ROTATION_LOCK from the accumulated product (vstab_set_partial_lock_fix)
    double cx, cy;               // working-size centre (rot_center, :1237)
};
void launch_smooth(const SmoothArgs& a, long call_first, int ncalls, WarpParams* out, cudaStream_t st);
// ORB / SIFT registration: fold one fit result into the "previously returned H" state (:724-787)
void launch_lock_update(const double* Tfit, const int* fit_counts, const int* nref, const int* ncur, const int* nmatch,
                        int reset, double* lock_h, int* tap, cudaStream_t st);
// offline ORB / SIFT: fold one fit result into reg[10] = {inverse(T), valid} (no carry: the carry is a scan at render time)
void launch_reg_store(const double* Tfit, const int* fit_counts, const int* nref, const int* ncur, const int* nmatch,
                      double* reg, cudaStream_t st);
// streaming ACCUMULATED_FULL_LOCK state update: acc <- T[p] * acc (src/stabilizer.cpp:334)
void launch_acc_update(const double* T, long t_mod, long p, int reset, double* acc_state, cudaStream_t st);
// offline: acc[k] for k in [a, a+n): acc[a] = I, acc[k] = T[k] * acc[k-1]
void launch_acc_scan(const double* T, long n_total, long anchor, double* acc, cudaStream_t st);

// ---------------------------------------------------------------- K16 auto-crop (vstab_set_crop)
struct CropArgs {
    double max_zoom, release;    // crop on: 1 < max_zoom <= 4, release > 0
    int R;                       // ceil((max_zoom - 1) / release): calls a need stays in the zoom of later calls
    int rows, cols;              // full-resolution frame
    double* need;                // n_j of call j at need[(j - need_base) % need_mod]
    long need_base, need_mod;
    int reset;                   // set need[0 .. need_mod) to 1 first (streaming: the calls before the enabling call)
};
// n_j for the nhalo calls before call_first (warp parameters in `halo`, read only) and for calls [call_first, +n) (in wp);
// then z_c for every call of wp, whose Hs / Minv become Z(z_c) * Hs and its inverse.
void launch_crop(const CropArgs& a, const WarpParams* halo, int nhalo, WarpParams* wp, long call_first, int n, cudaStream_t st);

// ---------------------------------------------------------------- K7 warpPerspective + border
void launch_warp(const uint8_t* frames, size_t pitch, size_t frame_stride, long slot_mod,
                 const WarpParams* wp, int nout, int w, int h,
                 uint8_t* out, size_t out_pitch, size_t out_frame_stride, cudaStream_t st,
                 unsigned long long* check = nullptr /* [nout], pre-zeroed: per-frame output checksum (warp.cu) */);

// ---------------------------------------------------------------- K15 YUV 4:2:0 <-> BGR (cv::cvtColor, bit-exact)
// the planes of one 4:2:0 frame relative to its base pointer; chroma sample k of a row is at off_u / off_v + k * cstep
struct YuvPlanes {
    size_t off_y, off_u, off_v;
    size_t step_y, step_u, step_v;
    int cstep;                   // 2: NV12 (one interleaved U,V plane, off_v = off_u + 1), 1: I420
};
// rows, cols even; frames `*_frame_stride` bytes apart (grid.z)
void launch_yuv420_to_bgr(const uint8_t* yuv, const YuvPlanes& L, size_t yuv_frame_stride, int nframes, int rows, int cols,
                          uint8_t* bgr, size_t pitch, size_t frame_stride, cudaStream_t st);
void launch_bgr_to_yuv420(const uint8_t* bgr, size_t pitch, size_t frame_stride, int nframes, int rows, int cols, uint8_t* yuv,
                          const YuvPlanes& L, size_t yuv_frame_stride, cudaStream_t st);

// ---------------------------------------------------------------- K14 feathered trail compositing (copyFeathered)
size_t trail_workspace_bytes(int w, int h, size_t frame_bytes);
// out = copyFeathered(frames[slot], bg, wp->Hs) (src/stabilizer.cpp:1051-1155); src_slot < 0: the slot named by *wp
void launch_trail(const uint8_t* frames, size_t pitch, size_t frame_stride, long slot_mod, const WarpParams* wp, int src_slot,
                  const uint8_t* bg, int w, int h, void* workspace, uint8_t* out, size_t out_pitch, cudaStream_t st);

// ---------------------------------------------------------------- K8 feature-path preprocessing
void build_nn_table(int src, int dst, int* host_tab);                       // cv::resize INTER_NEAREST offsets
size_t featprep_workspace_bytes(int w, int h);
// frame: device BGR (full resolution) -> out: device u8 w x h (tight), the conditioned working image
void launch_featprep(const uint8_t* frame, size_t pitch, const int* xofs, const int* yofs, int w, int h,
                     void* workspace, uint8_t* out, cudaStream_t st);


// ---------------------------------------------------------------- CUDA-graph replay of fixed launch sequences
// The ORB and SIFT front ends are long sequences of small dependent launches (44 / 119 per frame) whose arguments
// do not change from call to call in streaming.  The second call with the same arguments captures the sequence on
// its stream (thread-local capture) and every later one replays the graph: one launch, no per-kernel host cost,
// back-to-back scheduling on the device.
struct GraphCache {
    struct Entry { unsigned long long key[5]; cudaGraphExec_t exec; cudaGraph_t graph; int launches; int seen; };
    std::vector<Entry> entries;
    ~GraphCache();
};
// body(): enqueues the sequence on `st` (must be capturable: no allocation, no synchronisation)
template <class F>
void run_graphed(GraphCache& gc, const unsigned long long (&key)[5], cudaStream_t st, F&& body) {
    GraphCache::Entry* e = nullptr;
    for (auto& x : gc.entries) {
        bool same = true;
        for (int i = 0; i < 5; ++i) same = same && x.key[i] == key[i];
        if (same) { e = &x; break; }
    }
    if (!e) {
        if (gc.entries.size() >= 8) { body(); return; }
        GraphCache::Entry n{};
        for (int i = 0; i < 5; ++i) n.key[i] = key[i];
        gc.entries.push_back(n);
        body();                                     // first call: plain launches (also runs one-time attribute setup)
        return;
    }
    if (e->exec) { cudaGraphLaunch(e->exec, st); count_launch(e->launches); return; }
    if (e->seen < 0) { body(); return; }            // capture failed once: stay on plain launches
    const long long l0 = launch_count();
    if (cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal) != cudaSuccess) { cudaGetLastError(); e->seen = -1; body(); return; }
    body();
    cudaGraph_t g = nullptr;
    if (cudaStreamEndCapture(st, &g) != cudaSuccess || !g || cudaGraphInstantiate(&e->exec, g, 0) != cudaSuccess) {
        cudaGetLastError();
        if (g) cudaGraphDestroy(g);
        e->exec = nullptr; e->seen = -1;
        body();
        return;
    }
    e->graph = g;
    e->launches = (int)(launch_count() - l0);
    cudaGraphLaunch(e->exec, st);
}

// ---------------------------------------------------------------- K9 ORB, K10 Hamming matcher
constexpr int kOrbLevels = 12;             // ORB::create nlevels, src/stabilizer.cpp:485
constexpr int kOrbMaxKp = 4096;            // 2500 requested + retainBest ties, rounded up
struct OrbKeypoint { float x, y, size, angle, response; int octave; };     // cv::KeyPoint fields the path uses
struct OrbPlan {
    int w = 0, h = 0, max_kp = 0, cap = 0, ntiles = 0;
    size_t pyr_bytes = 0, cub_bytes = 0;
    void* levels = nullptr;                // OrbLevels (orb.cu)
    void* mem = nullptr;
    int2* tabs = nullptr;
    std::vector<size_t> tab_off;
    uint8_t *pyr = nullptr, *blur = nullptr, *score = nullptr;
    unsigned long long *cand = nullptr, *cand_sorted = nullptr;
    unsigned int* hist = nullptr;
    int* counters = nullptr;
    void* cub_temp = nullptr;
    GraphCache graphs;
};
// size_ratio: the reference's filterKeypointByRelativeSize ratio (0.10 for ORB; <= 0 keeps every level)
OrbPlan* orb_plan_create(int w, int h, double size_ratio, int max_keypoints, std::string* err);
void orb_plan_destroy(OrbPlan* P);
int orb_levels_used(const OrbPlan* P);
void launch_orb(OrbPlan* P, const uint8_t* gray, OrbKeypoint* kps, uint8_t* desc, int* count, bool reference_order,
                cudaStream_t st);
void launch_hamming_match(const uint8_t* ref_desc, const int* nref, const OrbKeypoint* ref_kps, const uint8_t* cur_desc,
                          const int* ncur, const OrbKeypoint* cur_kps, int max_kp, float ratio, int* best_idx, int* best_d,
                          int* second_d, uint8_t* good, float2* ref_pts, float2* cur_pts, uint8_t* status, int* nmatch,
                          cudaStream_t st);

// ---------------------------------------------------------------- K11 SIFT
constexpr int kSiftMaxOctaves = 12;
struct SiftPlan {
    int w = 0, h = 0, max_kp = 0, cand_cap = 0, kp_cap = 0;
    float max_size = 0.f;                  // relative-size filter of the reference (0.05 * rows), 0 = off
    size_t pyr_floats = 0, cub_bytes = 0;
    int radii[8] = {};
    void* octaves = nullptr;               // SiftOctaves (sift.cu)
    void* mem = nullptr;
    float* pyr = nullptr;
    unsigned long long *cand = nullptr, *keys = nullptr, *keys_sorted = nullptr;
    void* kps = nullptr;
    int *idx = nullptr, *idx_sorted = nullptr, *counters = nullptr;
    unsigned int *rkeys = nullptr, *rkeys_sorted = nullptr;
    uint8_t* alive = nullptr;
    void* cub_temp = nullptr;
    cudaStream_t aux[2] = {nullptr, nullptr};          // octaves >= 1 run beside the tail of the octave above them
    cudaEvent_t ev_g3[kSiftMaxOctaves] = {};           // Gaussian[kLayers] of octave o is ready (the next octave's base)
    cudaEvent_t ev_join[2] = {nullptr, nullptr};
    GraphCache graphs;
};
SiftPlan* sift_plan_create(int w, int h, double size_ratio, int max_keypoints, std::string* err);
void sift_plan_destroy(SiftPlan* P);
// octave count; w[o], h[o] and the float offset of Gaussian 0 of octave o in P->pyr (Gaussian i at off[o] + i * w * h)
int sift_plan_geometry(const SiftPlan* P, int* w, int* h, size_t* off /* or null */);
// the DoG extrema pass alone on whatever P->pyr holds (tests): candidates in P->cand, their count in P->counters[0]
void launch_sift_extrema(SiftPlan* P, cudaStream_t st);
// gray: device u8 w x h.  kps_out[max_kp] {x, y, size, angle, response, packed octave}, desc[max_kp][128] u8
void launch_sift(SiftPlan* P, const uint8_t* gray, OrbKeypoint* kps_out, uint8_t* desc, int* count, cudaStream_t st);

// ---------------------------------------------------------------- K12 exact L2 matcher (tcgen05)
// descriptors: u8 [n][128] (SIFT descriptors are integers 0..255).  best_d2 = exact squared distances.
// scratch: l2_match_scratch_bytes(max_kp, 1) device bytes.  The current rows beyond *ncur up to the next multiple of 128 are zeroed.
// Both return false, having launched nothing, when the driver's tensor-map encoder (cuTensorMapEncodeTiled) is missing or
// rejects the descriptor arrays.
size_t l2_match_scratch_bytes(int max_kp, int nframes);
bool launch_l2_match(const uint8_t* ref_desc, const int* nref, const OrbKeypoint* ref_kps, uint8_t* cur_desc,
                     const int* ncur, const OrbKeypoint* cur_kps, int max_kp, void* scratch, int* best_idx, int* best_d2, uint8_t* good,
                     float2* ref_pts, float2* cur_pts, uint8_t* status, int* nmatch, cudaStream_t st);
// the nearest-neighbour search alone, `nframes` current sets (cur_desc + f * max_kp * 128, ncur[f]) against one reference set
bool launch_l2_nn_batch(const uint8_t* ref_desc, const int* nref, uint8_t* cur_desc, const int* ncur, int max_kp, int nframes,
                        void* scratch, int* best_idx, int* best_d2, cudaStream_t st);

// ---------------------------------------------------------------- K13 simulator render
struct RenderPose { double R[9]; double cam[3]; };
void launch_render(const uint8_t* tex, int tex_rows, int tex_cols, const RenderPose* poses_dev, int n,
                   int w, int h, double focal, uint8_t* out, size_t pitch, size_t frame_stride,
                   cudaStream_t st, const double* rays = nullptr /* [3][h][w] from launch_render_rays, or null */,
                   const unsigned* tex4 = nullptr /* the texture as B G R x words from launch_render_tex4, or null */);
// the texture repacked to one 32-bit word per texel (one load per pixel instead of three)
void launch_render_tex4(const uint8_t* tex, int tex_rows, int tex_cols, unsigned* tex4, cudaStream_t st);
// the pose-independent camera rays of every pixel (24 bytes per pixel), for jobs that render many frames
void launch_render_rays(int w, int h, double focal, double* rays, cudaStream_t st);

}  // namespace vstabk
