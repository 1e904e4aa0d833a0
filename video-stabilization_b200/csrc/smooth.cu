// K6: sliding-window trajectory smoothing, full-lock accumulation, mode selection and the
// per-call warp parameters.
//   calculateGlobalSmoothingStabilization  /root/reference/src/stabilizer.cpp:793-852
//   calculateFullLockStabilization (ACCUMULATED branch)            :317-338, :438
//   mode switch + translation rescale                              :1231-1296
//   border colour 0.5 * cv::mean(presentation frame)               :1309
// Index algebra (SURVEY Appendix C): call c (>= 1) sees frames [lo, c], lo = max(0, c-W+1),
// presents p = max(0, c-F); window transforms are T[lo+1 .. c] with T[k] mapping k-1 -> k.
//   past   terms k = 1..p-lo      : A_k = inv(T[p-k+1]) * A_{k-1}
//   future terms r = 1..c-1-p     : B_r = B_{r-1} * T[p+r]      (newest transform excluded)
//   H = (sum A + sum B) / count   (no identity term; count==0 or non-finite -> I)
// Reference quirks kept on purpose: see SURVEY Appendix B.2-B.4, B.7, B.8.
// One warp per call: lane 0 walks the past chain, lane 1 the future chain (reference order).
#include "homography.cuh"
#include "kernels.h"

namespace vstabk {
namespace {

constexpr int kSmoothMaxTerms = 256;         // window terms staged in shared memory (18 KB); longer windows read global memory

VSTAB_D const double* t_at(const SmoothArgs& a, long k) { return a.T + (size_t)(k % a.t_mod) * 9; }

__global__ void __launch_bounds__(32)
smooth_kernel(SmoothArgs a, long call_first, int ncalls, WarpParams* __restrict__ out) {
    const int ci = blockIdx.x;
    if (ci >= ncalls) return;
    const int lane = threadIdx.x;
    const long c = call_first + ci;
    const long W = (long)a.P + 1 + a.F;
    const long lo = c - W + 1 > 0 ? c - W + 1 : 0;
    const long p = c - a.F > 0 ? c - a.F : 0;

    // lock modes before their lock call still present the window average (mode 5)
    int mode = a.mode;
    if ((mode == 0 || mode == 1 || mode == 2) && c < a.lock_call) mode = 5;

    double sum[9];
    for (int i = 0; i < 9; ++i) sum[i] = 0.0;
    int count = 0;
    // The window's transforms are staged in shared memory (the chains below would otherwise pay a global-memory
    // round trip per term) and the past ones are inverted in parallel, one matrix per lane at a time; the two
    // chains themselves stay sequential in the reference's order (lane 0: past, lane 1: future).
    __shared__ double sT[kSmoothMaxTerms][9];
    const long npast = p - lo, nfut = c - 1 - p > 0 ? c - 1 - p : 0;
    const bool staged = npast + nfut <= kSmoothMaxTerms;
    if (mode == 5 && staged) {
        for (long t = lane; t < npast + nfut; t += 32) {
            // slot t < npast: inverse of T[p - t]; slot npast + r: T[p + 1 + r]
            const double* src = t < npast ? t_at(a, p - t) : t_at(a, p + 1 + (t - npast));
            double m[9];
            for (int i = 0; i < 9; ++i) m[i] = src[i];
            if (t < npast) invert3(m, sT[t]);
            else for (int i = 0; i < 9; ++i) sT[t][i] = m[i];
        }
        __syncwarp();
    }
    if (mode == 5) {
        if (lane == 0) {
            double acc[9], inv[9], tmp[9];
            eye3(acc);
            for (long k = p; k > lo; --k) {                 // T[p], T[p-1], ..., T[lo+1]
                if (staged) for (int i = 0; i < 9; ++i) inv[i] = sT[p - k][i];
                else invert3(t_at(a, k), inv);
                matmul3(inv, acc, tmp);
                for (int i = 0; i < 9; ++i) { acc[i] = tmp[i]; sum[i] += tmp[i]; }
                ++count;
            }
        } else if (lane == 1) {
            double acc[9], tmp[9], cur[9];
            eye3(acc);
            for (long k = p + 1; k <= c - 1; ++k) {         // T[p+1] ... T[c-1]
                const double* src = staged ? sT[npast + (k - p - 1)] : t_at(a, k);
                for (int i = 0; i < 9; ++i) cur[i] = src[i];
                matmul3(acc, cur, tmp);
                for (int i = 0; i < 9; ++i) { acc[i] = tmp[i]; sum[i] += tmp[i]; }
                ++count;
            }
        }
    }
    // combine: avg = past_sum + future_sum (the reference adds past terms first)
    double fut[9];
    for (int i = 0; i < 9; ++i) fut[i] = __shfl_sync(0xffffffffu, sum[i], 1);
    const int fcount = __shfl_sync(0xffffffffu, count, 1);
    if (lane != 0) return;

    double Hs[9];
    eye3(Hs);
    const int total = count + fcount;
    if (total > 0) {
        double avg[9];
        // past partial sums were accumulated first, future terms added one by one after them;
        // adding the future block as one sum differs from the reference by O(1 ulp).
        for (int i = 0; i < 9; ++i) avg[i] = (sum[i] + fut[i]) / (double)total;
        if (finite9(avg))
            for (int i = 0; i < 9; ++i) Hs[i] = avg[i];
    }

    // ---- full-lock transform -------------------------------------------------------------
    double Hl[9];
    eye3(Hl);
    const bool partial = a.partial_fix && (mode == 3 || mode == 4);
    if (mode == 0 || partial) {
        const double* accp = a.acc + (size_t)(a.acc_mod > 0 ? (p % a.acc_mod) : 0) * 9;
        invert3(accp, Hl);                                // accumulatedTransform_.H.inv(), :438
        HParams hp;
        if (!decompose_h(Hl, 0.0, 0.0, &hp)) { eye3(Hl); hp.theta = 0.0; }   // :1240-1244
        if (partial) {
            // :1246-1260 as written, fed with the accumulated lock instead of the identity the reference's
            // calculateFullLockStabilization returns in these modes (the @todo of include/stabilizer.hpp:23):
            // R = getRotationMatrix2D(rot_center, theta in degrees, 1), H_translation_lock = R * H_lock (the accumulated
            // rotation is put back, the translation stays locked), H_rotation_lock = R^-1 (only the rotation is cancelled)
            // cv::getRotationMatrix2D: angle *= CV_PI / 180 (one constant), alpha = cos, beta = sin, Point2f centre
            const double kDegToRad = 3.1415926535897932384626433832795 / 180.0;
            const double ang = (hp.theta * 180.0 / 3.14159265358979323846) * kDegToRad;
            const double al = cos(ang), be = sin(ang);
            double R[9] = {al, be, (1.0 - al) * a.cx - be * a.cy, -be, al, be * a.cx + (1.0 - al) * a.cy, 0.0, 0.0, 1.0};
            double tmp[9];
            if (mode == 3) matmul3(R, Hl, tmp);
            else invert3(R, tmp);
            for (int i = 0; i < 9; ++i) Hl[i] = tmp[i];
        }
    }
    if ((mode == 1 || mode == 2) && a.reg) {
        // offline: the matrix returned at call c is the registration of the latest presented frame that
        // produced one (the reference's "previously returned H" carry, :446), identity at the capture call
        if (c > a.lock_call)
            for (long q = p; q >= a.reg_lo; --q)
                if (a.reg[(size_t)q * 10 + 9] != 0.0) { for (int i = 0; i < 9; ++i) Hl[i] = a.reg[(size_t)q * 10 + i]; break; }
        HParams hp;
        if (!decompose_h(Hl, 0.0, 0.0, &hp)) eye3(Hl);    // :1240-1244
    } else if ((mode == 1 || mode == 2) && a.lock_h) {    // ORB / SIFT registration (:440-787)
        for (int i = 0; i < 9; ++i) Hl[i] = a.lock_h[i];
        HParams hp;
        if (!decompose_h(Hl, 0.0, 0.0, &hp)) eye3(Hl);    // :1240-1244
    }
    double H[9];
    if (mode == 5) { for (int i = 0; i < 9; ++i) H[i] = Hs[i]; }
    else if (mode == 0 || mode == 1 || mode == 2 || partial) { for (int i = 0; i < 9; ++i) H[i] = Hl[i]; }
    else { eye3(H); }                                     // T/R lock: identity (SURVEY B.7)

    WarpParams wp;
    for (int i = 0; i < 9; ++i) wp.Hw[i] = H[i];
    if (fabs(a.scale - 1.0) > 1e-6) {                     // :1291-1296
        H[2] /= a.scale;
        H[5] /= a.scale;
    }
    for (int i = 0; i < 9; ++i) wp.Hs[i] = H[i];
    invert3(H, wp.Minv);
    const long slot = a.sums_mod > 0 ? (p % a.sums_mod) : (p - a.frame_base);
    wp.src_slot = (int)slot;
    // no sums: the matrices alone are wanted (auto-crop's halo calls, whose presentation frames another chunk holds)
    for (int ch = 0; ch < 3 && a.sums; ++ch) {
        const double mean = (double)a.sums[(size_t)slot * 3 + ch] / a.npix;   // cv::mean
        int v = __double2int_rn(0.5 * mean);                                  // saturate_cast<uchar>
        v = v < 0 ? 0 : (v > 255 ? 255 : v);
        wp.border[ch] = (unsigned char)v;
    }
    if (!a.sums) wp.border[0] = wp.border[1] = wp.border[2] = 0;
    wp.border[3] = 0;
    out[ci] = wp;
}

// ORB / SIFT registration result -> the matrix calculateFullLockStabilization returns (:724-787):
// a valid fit of >= 10 matches between >= 10 keypoints on either side replaces the previously
// returned matrix by inverse(H with scale forced to 1); anything else keeps it.  reset: reference
// capture (:520-589) returns identity and resets the fallback (:528).
__global__ void lock_update_kernel(const double* __restrict__ Tfit, const int* __restrict__ fit_counts,
                                   const int* __restrict__ nref, const int* __restrict__ ncur,
                                   const int* __restrict__ nmatch, int reset, double* __restrict__ lock_h,
                                   int* __restrict__ tap /* {ncur, nref, nmatch, inliers, updated} or null */) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    if (reset) {
        eye3(lock_h);
        if (tap) { tap[0] = *nref; tap[1] = *nref; tap[2] = 0; tap[3] = 0; tap[4] = 0; }
        return;
    }
    bool ok = *ncur >= kMinPointsForMotion && *nref >= kMinPointsForMotion && *nmatch >= kMinPointsForMotion &&
              fit_counts[1] > 0;
    double inv[9];
    if (ok) ok = invert3(Tfit, inv) && finite9(inv);
    if (ok) for (int i = 0; i < 9; ++i) lock_h[i] = inv[i];
    if (tap) { tap[0] = *ncur; tap[1] = *nref; tap[2] = *nmatch; tap[3] = fit_counts[1]; tap[4] = ok ? 1 : 0; }
}

__global__ void reg_store_kernel(const double* __restrict__ Tfit, const int* __restrict__ fit_counts,
                                 const int* __restrict__ nref, const int* __restrict__ ncur,
                                 const int* __restrict__ nmatch, double* __restrict__ reg) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    bool ok = *ncur >= kMinPointsForMotion && *nref >= kMinPointsForMotion && *nmatch >= kMinPointsForMotion &&
              fit_counts[1] > 0;
    double inv[9];
    if (ok) ok = invert3(Tfit, inv) && finite9(inv);
    if (!ok) eye3(inv);
    for (int i = 0; i < 9; ++i) reg[i] = inv[i];
    reg[9] = ok ? 1.0 : 0.0;
}

// acc <- T[p] * acc   (or identity on the first call after setStabilizationMode)
__global__ void acc_update_kernel(const double* T, long t_mod, long p, int reset, double* acc) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    if (reset) { eye3(acc); return; }
    double tmp[9];
    matmul3(T + (size_t)(p % t_mod) * 9, acc, tmp);
    for (int i = 0; i < 9; ++i) acc[i] = tmp[i];
}

// ---- offline prefix product: acc[k] = T[k] * acc[k-1], acc[anchor] = I (acc_seq_kernel below) ----------
constexpr int kScanChunk = 256;

}  // namespace

void launch_smooth(const SmoothArgs& a, long call_first, int ncalls, WarpParams* out, cudaStream_t st) {
    if (ncalls <= 0) return;
    count_launch(1);
    smooth_kernel<<<ncalls, 32, 0, st>>>(a, call_first, ncalls, out);
}

void launch_lock_update(const double* Tfit, const int* fit_counts, const int* nref, const int* ncur, const int* nmatch,
                        int reset, double* lock_h, int* tap, cudaStream_t st) {
    count_launch(1);
    lock_update_kernel<<<1, 32, 0, st>>>(Tfit, fit_counts, nref, ncur, nmatch, reset, lock_h, tap);
}

void launch_reg_store(const double* Tfit, const int* fit_counts, const int* nref, const int* ncur, const int* nmatch,
                      double* reg, cudaStream_t st) {
    count_launch(1);
    reg_store_kernel<<<1, 32, 0, st>>>(Tfit, fit_counts, nref, ncur, nmatch, reg);
}

void launch_acc_update(const double* T, long t_mod, long p, int reset, double* acc_state, cudaStream_t st) {
    count_launch(1);
    acc_update_kernel<<<1, 32, 0, st>>>(T, t_mod, p, reset, acc_state);
}

namespace {
// The accumulated-lock prefix acc[k] = T[k] * acc[k-1] (acc[anchor] = I) as ONE strictly sequential chain in the reference's
// own order (src/stabilizer.cpp:334: `acc <- T[p-1] * acc` once per call): products of 3x3 doubles do not associate bit for
// bit, and a chunked scan (reduce / scan / apply, round 1) re-associates them across chunk boundaries, so a 2000-frame offline
// clip and the streaming calls would differ in the last bits.  One thread walks the chain; the CTA stages 256 transforms at
// a time through shared memory and writes the running products back coalesced.  ~50 ns per frame: 0.03 ms for the bench's 512
// frames (the three-kernel scan took 0.06 ms), 5 ms for 100 000.
__global__ void __launch_bounds__(128)
acc_seq_kernel(const double* __restrict__ T, long n_total, long anchor, double* __restrict__ acc_out) {
    __shared__ double sT[kScanChunk * 9];
    __shared__ double run[9];
    if (threadIdx.x == 0) { eye3(run); if (anchor < n_total) eye3(acc_out + (size_t)anchor * 9); }
    for (long k0 = anchor + 1; k0 < n_total; k0 += kScanChunk) {
        const long k1 = k0 + kScanChunk < n_total ? k0 + kScanChunk : n_total;
        __syncthreads();
        for (long i = threadIdx.x; i < (k1 - k0) * 9; i += blockDim.x) sT[i] = T[(size_t)k0 * 9 + i];
        __syncthreads();
        if (threadIdx.x == 0) {
            double a[9], tmp[9];
            for (int i = 0; i < 9; ++i) a[i] = run[i];
            for (long k = k0; k < k1; ++k) {
                matmul3(sT + (size_t)(k - k0) * 9, a, tmp);
                for (int i = 0; i < 9; ++i) { a[i] = tmp[i]; sT[(size_t)(k - k0) * 9 + i] = tmp[i]; }
            }
            for (int i = 0; i < 9; ++i) run[i] = a[i];
        }
        __syncthreads();
        for (long i = threadIdx.x; i < (k1 - k0) * 9; i += blockDim.x) acc_out[(size_t)k0 * 9 + i] = sT[i];
    }
}

}  // namespace

void launch_acc_scan(const double* T, long n_total, long anchor, double* acc, cudaStream_t st) {
    if (anchor >= n_total) return;
    count_launch(1);
    acc_seq_kernel<<<1, 128, 0, st>>>(T, n_total, anchor, acc);
}

}  // namespace vstabk
