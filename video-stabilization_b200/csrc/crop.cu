// K16: auto-crop (vstab_set_crop).  Per call c: the zoom n_c its own warp needs to show no border (crop_need,
// homography.cuh), the causal schedule z_c = clamp(max_{j in [max(0, c-R), c]} (n_j - (c-j) * release), 1, max_zoom), and
// the matrix the warp / trail then apply, Hc = Z(z_c) * H_stabilize_scaled.  The schedule reads the needs of the R calls
// before c from a per-call history, so its bits do not depend on how calls are cut into batches or shards.
// Built without FMA contraction: every term is n_j - (double)(c - j) * release as written, and max is exact.
#include "homography.cuh"
#include "kernels.h"

namespace vstabk {
namespace {

constexpr int kCropThreads = 256;

VSTAB_D long need_slot(const CropArgs& a, long j) { return (j - a.need_base) % a.need_mod; }

// One CTA: (0) optional reset of the history, (1) the needs of halo + batch, (2) one warp per call for the schedule.
__global__ void __launch_bounds__(kCropThreads)
crop_kernel(CropArgs a, const WarpParams* __restrict__ halo, int nhalo, WarpParams* __restrict__ wp, long call_first, int n) {
    if (a.reset)
        for (long i = threadIdx.x; i < a.need_mod; i += blockDim.x) a.need[i] = 1.0;
    __syncthreads();
    for (int i = threadIdx.x; i < nhalo + n; i += blockDim.x) {
        const double* H = i < nhalo ? halo[i].Hs : wp[i - nhalo].Hs;
        a.need[need_slot(a, call_first - nhalo + i)] = crop_need(H, a.rows, a.cols, a.max_zoom);
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int ci = warp; ci < n; ci += kCropThreads / 32) {
        const long c = call_first + ci;
        const long lo = c - a.R > 0 ? c - a.R : 0;
        double m = 1.0;
        for (long j = lo + lane; j <= c; j += 32) {
            const double v = a.need[need_slot(a, j)] - (double)(c - j) * a.release;
            m = fmax(m, v);
        }
        for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
        if (lane == 0) {
            const double z = m > a.max_zoom ? a.max_zoom : m;     // m >= 1
            double H[9], Hc[9];
            for (int i = 0; i < 9; ++i) H[i] = wp[ci].Hs[i];
            crop_apply(z, H, a.rows, a.cols, Hc);
            for (int i = 0; i < 9; ++i) wp[ci].Hs[i] = Hc[i];
            invert3(Hc, wp[ci].Minv);                              // the inversion smooth_kernel applies to Hs
        }
    }
}

}  // namespace

void launch_crop(const CropArgs& a, const WarpParams* halo, int nhalo, WarpParams* wp, long call_first, int n, cudaStream_t st) {
    if (n <= 0) return;
    count_launch(1);
    crop_kernel<<<1, kCropThreads, 0, st>>>(a, halo, nhalo, wp, call_first, n);
}

}  // namespace vstabk
