// K3: Shi-Tomasi corners = cv::goodFeaturesToTrack(gray, 1300, 0.01, minDist, noMask, 3, 3, false, 0.04)
// (/root/reference/src/stabilizer.cpp:931-980; the reference calls it twice with identical
// output, :949 and :961 -- it runs once here).  SURVEY A.5:
//   pass A  cornerMinEigenVal: Sobel3 (OpenCV's FMA order) -> products -> 3x3 box (f64 sums)
//           -> min eigenvalue (f32), global max, and -- in the same kernel -- every 3x3 local
//           maximum as a 64-bit sort key (value desc, address desc).  OpenCV thresholds at
//           0.01*max *before* its dilate test, but a pixel above the threshold can only lose to
//           a neighbour that is itself above it, so "local maximum" does not depend on the
//           threshold: the cut is applied after the sort, where it is a prefix of the list.
//           The min-eigenvalue map is not written to HBM (only when a tap asks for it).
//   sort    segmented radix sort of the candidate keys (one segment per frame);
//   pass C  greedy min-distance suppression in sorted order on a cell grid held in shared
//           memory, one warp per frame, 32 candidates per step with ballot/shuffle conflict
//           resolution -- the accepted set and its order equal the sequential OpenCV loop.
#include <type_traits>
#include <cub/block/block_radix_sort.cuh>
#include <cub/device/device_segmented_radix_sort.cuh>
#include "kernels.h"

namespace vstabk {
namespace {

constexpr unsigned short kEmpty16 = 0xffffu;
constexpr int kCellCap = 4;                       // u16 slots per cell ({dy,dx} relative to the cell)
constexpr int kGreedySmemMax = 200 * 1024;

// Pass A as a register/shuffle stream, no shared memory: one warp owns a strip of kStripW = 28 columns and
// marches down a segment of kSegH rows.  Lane l holds the derivative products of column sx0-2+l (reflected into
// the image like cv::boxFilter's BORDER_REFLECT_101 does with the covariance images); the horizontal 3-sums come
// from shfl.down on the f64 products, the vertical 3-sums from the last three rows kept in registers (f64, the
// order of OpenCV's row/column sums), the eigenvalue row from those, and the 3x3 local-maximum test from the last
// three eigenvalue rows (horizontal neighbours by shuffle).  Each gray row is read once per strip (+4 halo
// columns, +4 halo rows per segment); every f32 product is converted to f64 once.
constexpr int kStripW = 28, kSegH = 90, kEigWarps = 4;   // (segment height 45 / 60 / 90 / 120 / 180: 0.663 / 0.655 / 0.646 / 0.658 / 0.670 ms)
constexpr int kEigPrefetchRows = 4;                      // eig_kernel's `pf`: L1 prefetch distance in rows

struct D3 { double xx, xy, yy; };

__global__ void __launch_bounds__(32 * kEigWarps, 8)
eig_kernel(const uint8_t* __restrict__ gray, size_t gray_stride, int w, int h, int nstrips, int nsegs, int seg_h, int idx_bits,
           float* __restrict__ eig_out, unsigned int* __restrict__ maxbits,
           unsigned long long* __restrict__ keys, int* __restrict__ seg_end, int cap, double quality, int pf) {
    const int lane = threadIdx.x & 31;
    const int item = blockIdx.x * kEigWarps + (threadIdx.x >> 5);
    const int frame = blockIdx.y;
    if (item >= nstrips * nsegs) return;
    const int seg = item / nstrips, strip = item - seg * nstrips;
    const int sx0 = strip * kStripW;
    const int ya = seg * seg_h, yb = min(ya + seg_h, h);
    const uint8_t* src = gray + (size_t)frame * gray_stride;

    // scale = 1 / (2^(ksize-1) * blockSize * 255) ; k1 = float(scale), k0 = float(2*scale)
    const float k1 = (float)(1.0 / (4.0 * 3.0 * 255.0));
    const float k0 = (float)(2.0 / (4.0 * 3.0 * 255.0));
    // this lane's product column, reflected into the image, and its Sobel taps (BORDER_REFLECT_101 of the gray image)
    const int xr = reflect101(min(sx0 - 2 + lane, w + 1), w);
    const int cm = reflect101(xr - 1, w), cp = reflect101(xr + 1, w);
    // OpenCV's row filter runs its FMA vector body over the first floor(w/32)*32 columns and a scalar,
    // un-contracted tail over the rest ([probe] cv2 4.13.0 on AVX-512 hosts; all production widths
    // 640/1280/1920/3840 are multiples of 32 and never reach the tail).
    const bool fma_col = xr < (w & ~31);
    // S = p[x+1] - p[x-1] (Dx row term), R = k1 p[x-1] + k0 p[x] + k1 p[x+1] (Dy row term) of a gray row; the three
    // bytes of a row are fetched one row ahead of their use (load_raw / row_terms), so the loop never waits for them
    auto load_raw = [&](int y, unsigned& a, unsigned& b, unsigned& c) {
        const int ro = y * w;                                    // (a working image has far fewer than 2^31 pixels)
        a = __ldg(src + (ro + cm)); b = __ldg(src + (ro + xr)); c = __ldg(src + (ro + cp));
    };
    auto row_terms = [&](unsigned a, unsigned b, unsigned c, float& S, float& R) {
        const float gm = (float)a, g0 = (float)b, gp = (float)c;
        S = __fsub_rn(gp, gm);
        R = fma_col ? __fmaf_rn(gp, k1, __fmaf_rn(g0, k0, __fmul_rn(gm, k1)))
                    : __fadd_rn(__fadd_rn(__fmul_rn(gm, k1), __fmul_rn(g0, k0)), __fmul_rn(gp, k1));
    };
    auto load_row = [&](int y, float& S, float& R) {
        unsigned a, b, c;
        load_raw(y, a, b, c);
        row_terms(a, b, c, S, R);
    };

    const int xe = sx0 - 1 + lane;                              // eigenvalue column of this lane (lanes 0..29)
    const bool e_valid = lane < 30 && xe >= 0 && xe < w;
    const bool own_col = lane >= 1 && lane <= kStripW && xe < w;
    const bool cand_col = own_col && xe >= 1 && xe < w - 1;
    const int ye_lo = max(ya - 1, 0), ye_hi = min(yb, h - 1);   // eigenvalue rows this segment needs
    const int p_lo = max(ye_lo - 1, 0), p_hi = min(ye_hi + 1, h - 1);   // product rows (all inside the image)
    const int yc_lo = max(ya, 1), yc_hi = min(yb, h - 1);       // candidate rows [yc_lo, yc_hi)

    // rolling state, indexed by compile-time slots (the row loop is unrolled by 3, so nothing is ever moved):
    // gray row g -> slot (g - p_lo + 1) % 3; product row yp -> slot j = (yp - p_lo) % 3; eigenvalue row yp-1 -> slot j
    float S[3], R[3];
    D3 RS[3] = {{0.0, 0.0, 0.0}, {0.0, 0.0, 0.0}, {0.0, 0.0, 0.0}};   // horizontal 3-sums of the product rows
    float E[3] = {0.f, 0.f, 0.f}, HM[3] = {0.f, 0.f, 0.f}, H3[3] = {0.f, 0.f, 0.f};   // eig row: value, max(left,right), 3-max
    load_row(reflect101(p_lo - 1, h), S[0], R[0]);
    load_row(p_lo, S[1], R[1]);
    unsigned ra, rb, rc;                                        // raw bytes of gray row yp + 1
    load_raw(reflect101(p_lo + 1, h), ra, rb, rc);
    float vmax = 0.f;
    // candidates must exceed this (0: the eigenvalue must be positive)
    float cut = (float)((double)__uint_as_float(*(volatile unsigned int*)(maxbits + frame)) * quality) * 0.999f;
    __shared__ unsigned long long queue_all[kEigWarps][64];
    unsigned long long* queue = queue_all[threadIdx.x >> 5];
    int qn = 0;
    // One row of the stream.  kSteady: a row away from every boundary of the segment and of the image -- all the range tests
    // below are known true at compile time, the next gray row needs no reflection -- which is every row but the first and last
    // few of a segment; the generic instance keeps the tests.  j: the compile-time slot of product row yp.
    auto step = [&](auto steady_c, auto j_c, const int yp) {
        constexpr bool kSteady = decltype(steady_c)::value;
        constexpr int j = decltype(j_c)::value, jA = (j + 1) % 3, jB = (j + 2) % 3;   // slots of rows yp, yp-2, yp-1
        if (kSteady || yp <= p_hi) {
            row_terms(ra, rb, rc, S[jB], R[jB]);                 // gray row yp+1
            load_raw(kSteady ? yp + 2 : reflect101(yp + 2, h), ra, rb, rc);   // (h + 1 at most: still a valid reflection)
            // every row of the strip starts a new 128-byte line: ask for the line `pf` rows further down now
            if (pf > 0) asm volatile("prefetch.global.L1 [%0];" ::"l"(src + (min(yp + 2 + pf, h - 1) * w + xr)));
            // Dx = fma(S[y-1] + S[y+1], k1, S[y]*k0),  Dy = R[y+1] - R[y-1]
            const float dx = __fmaf_rn(__fadd_rn(S[j], S[jB]), k1, __fmul_rn(S[jA], k0));
            const float dy = __fsub_rn(R[jB], R[j]);
            const double pxx = (double)__fmul_rn(dx, dx), pxy = (double)__fmul_rn(dx, dy), pyy = (double)__fmul_rn(dy, dy);
            RS[j].xx = __dadd_rn(__dadd_rn(pxx, __shfl_down_sync(0xffffffffu, pxx, 1)), __shfl_down_sync(0xffffffffu, pxx, 2));
            RS[j].xy = __dadd_rn(__dadd_rn(pxy, __shfl_down_sync(0xffffffffu, pxy, 1)), __shfl_down_sync(0xffffffffu, pxy, 2));
            RS[j].yy = __dadd_rn(__dadd_rn(pyy, __shfl_down_sync(0xffffffffu, pyy, 1)), __shfl_down_sync(0xffffffffu, pyy, 2));
        } else {
            RS[j] = RS[jA];                                     // below the last image row: product row h == row h-2
        }
        const int ye = yp - 1;
        if (kSteady || (ye >= ye_lo && ye <= ye_hi)) {
            const D3 U = (!kSteady && ye == 0) ? RS[j] : RS[jA];   // above the first image row: product row -1 == row 1
            const double sxx = __dadd_rn(__dadd_rn(U.xx, RS[jB].xx), RS[j].xx);
            const double sxy = __dadd_rn(__dadd_rn(U.xy, RS[jB].xy), RS[j].xy);
            const double syy = __dadd_rn(__dadd_rn(U.yy, RS[jB].yy), RS[j].yy);
            const float a = __fmul_rn((float)sxx, 0.5f);
            const float b = (float)sxy;
            const float cc = __fmul_rn((float)syy, 0.5f);
            const float d = __fsub_rn(a, cc);
            const float rad = __fsqrt_rn(__fadd_rn(__fmul_rn(d, d), __fmul_rn(b, b)));
            const float e = e_valid ? __fsub_rn(__fadd_rn(a, cc), rad) : 0.f;
            if (own_col && (kSteady || (ye >= ya && ye < yb))) {
                vmax = fmaxf(vmax, e);
                if (eig_out) eig_out[(size_t)frame * w * h + (size_t)ye * w + xe] = e;
            }
            const float hm = fmaxf(__shfl_up_sync(0xffffffffu, e, 1), __shfl_down_sync(0xffffffffu, e, 1));
            E[j] = e; HM[j] = hm; H3[j] = fmaxf(hm, e);
            // 3x3 local maxima of row yc = ye - 1 (ties kept, like eig == dilate(eig)) inside the 1-px image border
            const int yc = ye - 1;
            if (kSteady || (yc >= yc_lo && yc < yc_hi)) {
                const float v = E[jB];
                // conservative early cut: the running maximum only grows, so anything at or below
                // 0.01 * (maximum seen so far) is certainly below the final threshold
                const bool is_cand = cand_col && v > cut && v >= HM[jB] && v >= H3[jA] && v >= H3[j];
                const unsigned ball = __ballot_sync(0xffffffffu, is_cand);
                if (ball) {
                    // append to this warp's queue; 32 keys leave with one atomic and one coalesced 256-byte store
                    if (is_cand)
                        queue[qn + __popc(ball & ((1u << lane) - 1u))] =
                            ((unsigned long long)__float_as_uint(v) << idx_bits) | (unsigned long long)(unsigned)(yc * w + xe);
                    qn += __popc(ball);
                    __syncwarp();
                    if (qn >= 32) {
                        int pos0 = 0;
                        if (lane == 0) pos0 = atomicAdd(seg_end + frame, 32);
                        pos0 = __shfl_sync(0xffffffffu, pos0, 0);
                        const unsigned long long k0 = queue[lane], k1 = queue[32 + lane];
                        if (pos0 + lane < (frame + 1) * cap) keys[pos0 + lane] = k0;
                        __syncwarp();
                        queue[lane] = k1;
                        qn -= 32;
                        __syncwarp();
                    }
                }
            }
        }
    };
    // generic row with the end-of-segment test; returns true when the segment is finished
    auto edge = [&](auto j_c, const int yp) -> bool {
        if (yp > p_hi + 1 || (yp > p_hi && p_hi != h - 1)) return true;
        step(std::false_type{}, j_c, yp);
        return false;
    };
    const std::integral_constant<int, 0> J0{};
    const std::integral_constant<int, 1> J1{};
    const std::integral_constant<int, 2> J2{};
    // steady rows: yp <= p_hi, yp + 2 <= h - 1, ye = yp - 1 in [max(ye_lo, 1), ye_hi] and in [ya, yb), yc = yp - 2 in [yc_lo, yc_hi)
    const int ys_lo = max(max(ye_lo + 1, 2), max(ya + 1, yc_lo + 2));
    const int ys_hi = min(min(p_hi, h - 3), min(min(ye_hi + 1, yb), yc_hi + 1));
    bool done = false;
    for (int yp0 = p_lo; !done; yp0 += 3) {
        if (yp0 >= ys_lo && yp0 + 2 <= ys_hi) {
            step(std::true_type{}, J0, yp0);
            step(std::true_type{}, J1, yp0 + 1);
            step(std::true_type{}, J2, yp0 + 2);
        } else {
            done = edge(J0, yp0);
            if (!done) done = edge(J1, yp0 + 1);
            if (!done) done = edge(J2, yp0 + 2);
        }
        // publish the running maximum every 12 rows (and at the end), and refresh the early cut from the frame's
        // maximum so far
        if (done || (yp0 - p_lo) % 12 == 9) {
            float m = vmax;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
            unsigned old = 0u;
            if (lane == 0) old = atomicMax(maxbits + frame, __float_as_uint(m));      // non-negative floats order like their bits
            old = __shfl_sync(0xffffffffu, old, 0);
            const float lb = fmaxf(__uint_as_float(old), m);
            cut = fmaxf(cut, (float)((double)lb * quality) * 0.999f);
        }
    }
    // flush the rest of the queue
    if (qn > 0) {
        int pos0 = 0;
        if (lane == 0) pos0 = atomicAdd(seg_end + frame, qn);
        pos0 = __shfl_sync(0xffffffffu, pos0, 0);
        if (lane < qn && pos0 + lane < (frame + 1) * cap) keys[pos0 + lane] = queue[lane];
    }
}

__global__ void gftt_reset_kernel(unsigned int* maxbits, int* seg_begin, int* seg_end, int cap, int nframes) {
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f < nframes) {
        maxbits[f] = 0u;
        seg_begin[f] = f * cap;
        seg_end[f] = f * cap;
    }
}

__global__ void clamp_segments_kernel(int* seg_end, int cap, int nframes) {
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f < nframes) seg_end[f] = min(seg_end[f], (f + 1) * cap);
}

// Greedy minimum-distance selection, one warp per frame (the other warps of the CTA only help to clear the grid).
// The cell grid (4 u16 slots per cell, {dy,dx} relative to the cell origin) lives in shared memory when it
// fits, else in the global scratch `grid_glob`.  32 candidates per step, in rank order:
//   1. every lane tests its candidate against the accepted points of the 3 x 3 cells around it (branch-free);
//   2. conflicts inside the batch: every surviving lane builds the mask of lower-ranked survivors closer than
//      min_distance, then
//      the accept / reject sets grow to their fixed point with two ballots per round (a lane is accepted once all
//      its conflicting lower lanes are rejected, rejected once one of them is accepted) -- the same set and order
//      as OpenCV's sequential loop, without a serial pass over the lanes;
//   3. accepted lanes append their point and register it in the grid.
constexpr int kGreedyThreads = 128;

// Steps 1-3 for the sorted candidates k[0..n) of one frame, executed by one warp; `accepted` carries over between
// chunks of the same frame.  Returns false once a candidate at or below the quality threshold shows up (everything
// after it is below, too).
VSTAB_D bool greedy_warp(const unsigned long long* __restrict__ k, int n, int idx_bits, float thr, int w, int min_distance,
                         int cell, int grid_w, int grid_h, unsigned short* gfr, int* bxy, int max_corners,
                         float2* __restrict__ out, int& accepted) {
    const int lane = threadIdx.x & 31;
    const int md2 = min_distance * min_distance;
    const unsigned lt = (1u << lane) - 1u;
    const unsigned long long idx_mask = (1ull << idx_bits) - 1ull;
    unsigned long long key_next = lane < n ? k[lane] : 0ull;
    for (int base = 0; base < n && accepted < max_corners; base += 32) {
        const int rank = base + lane;
        const unsigned long long key = key_next;
        if (rank + 32 < n) key_next = k[rank + 32];
        // THRESH_TOZERO cut: a prefix of the sorted list
        const bool valid = rank < n && __uint_as_float((unsigned)(key >> idx_bits)) > thr;
        if (!__any_sync(0xffffffffu, valid)) return false;
        const unsigned idx = (unsigned)(key & idx_mask);
        const int y = valid ? (int)(idx / (unsigned)w) : 0;
        const int x = valid ? (int)(idx - (unsigned)y * (unsigned)w) : 0;
        bool ok = valid;
        int cx = 0, cy = 0;
        if (min_distance >= 1) {
            cx = x / cell;
            cy = y / cell;
#pragma unroll
            for (int dy = -1; dy <= 1; ++dy)
#pragma unroll
                for (int dx = -1; dx <= 1; ++dx) {
                    const int gx = cx + dx, gy = cy + dy;
                    const bool inb = gx >= 0 && gx < grid_w && gy >= 0 && gy < grid_h;
                    const int gxc = min(max(gx, 0), grid_w - 1), gyc = min(max(gy, 0), grid_h - 1);
                    uint2 sl = *reinterpret_cast<const uint2*>(gfr + ((size_t)gyc * grid_w + gxc) * kCellCap);
                    if (!inb) sl = make_uint2(0xffffffffu, 0xffffffffu);
                    const unsigned s4[4] = {sl.x & 0xffffu, sl.x >> 16, sl.y & 0xffffu, sl.y >> 16};
                    const int ox = x - gxc * cell, oy = y - gyc * cell;
#pragma unroll
                    for (int q = 0; q < kCellCap; ++q) {
                        const int ddx = ox - (int)(s4[q] & 0xffu), ddy = oy - (int)(s4[q] >> 8);
                        if (s4[q] != kEmpty16 && ddx * ddx + ddy * ddy < md2) ok = false;
                    }
                }
            // conflicts inside the batch, resolved in rank order: one pass over the compact list of the survivors
            const unsigned okmask = __ballot_sync(0xffffffffu, ok);
            const int nok = __popc(okmask);
            if (ok) bxy[__popc(okmask & lt)] = x | (y << 12) | (lane << 24);     // (x, y < 4096)
            __syncwarp();
            unsigned cm = 0;
#pragma unroll 4
            for (int t = 0; t < nok; ++t) {
                const int o = bxy[t];
                const int ddx = x - (o & 0xfff), ddy = y - ((o >> 12) & 0xfff);
                if (ddx * ddx + ddy * ddy < md2) cm |= 1u << (o >> 24);
            }
            __syncwarp();
            cm &= lt;                                          // lower-ranked candidates that passed the grid test
            unsigned acc = 0, rej = ~okmask;
            for (;;) {
                acc |= __ballot_sync(0xffffffffu, ok && (cm & ~rej) == 0);
                rej |= __ballot_sync(0xffffffffu, ok && (cm & acc) != 0);
                if ((acc | rej) == 0xffffffffu) break;
            }
            ok = (acc >> lane) & 1u;
        }
        const unsigned accm = __ballot_sync(0xffffffffu, ok);
        const int my = accepted + __popc(accm & lt);
        if (ok && my < max_corners) {
            out[my] = make_float2((float)x, (float)y);
            if (min_distance >= 1) {
                unsigned short* cellp = gfr + ((size_t)cy * grid_w + cx) * kCellCap;
                const unsigned short val = (unsigned short)(((y - cy * cell) << 8) | (x - cx * cell));
                for (int q = 0; q < kCellCap; ++q)
                    if (atomicCAS(cellp + q, kEmpty16, val) == kEmpty16) break;
            }
        }
        accepted += __popc(accm);
        __syncwarp();
    }
    return true;
}

// Unfused schedule: the keys were sorted by cub (one segment per frame).
__global__ void __launch_bounds__(kGreedyThreads)
greedy_kernel(const unsigned long long* __restrict__ keys, const int* __restrict__ seg_begin,
              const int* __restrict__ seg_end, const unsigned int* __restrict__ maxbits, double quality, int idx_bits,
              int w, int min_distance, int cell, int grid_w, int grid_h,
              unsigned short* grid_glob, int use_smem, int max_corners,
              float2* __restrict__ pts, int* __restrict__ counts) {
    extern __shared__ unsigned short grid_sm[];
    __shared__ int bxy[32];
    const int frame = blockIdx.x;
    const int ncells = grid_w * grid_h;
    unsigned short* gfr = use_smem ? grid_sm : grid_glob + (size_t)frame * ncells * kCellCap;
    {
        uint2* g2 = reinterpret_cast<uint2*>(gfr);
        for (int i = threadIdx.x; i < ncells; i += kGreedyThreads) g2[i] = make_uint2(0xffffffffu, 0xffffffffu);
    }
    __syncthreads();
    if (threadIdx.x >= 32) return;
    const float thr = (float)((double)__uint_as_float(maxbits[frame]) * quality);       // cv::threshold takes float(thresh)
    int accepted = 0;
    greedy_warp(keys + seg_begin[frame], seg_end[frame] - seg_begin[frame], idx_bits, thr, w, min_distance, cell, grid_w,
                grid_h, gfr, bxy, max_corners, pts + (size_t)frame * kMaxCorners, accepted);
    if ((threadIdx.x & 31) == 0) counts[frame] = min(accepted, max_corners);
}

// Fused schedule (the default): one CTA per frame selects, sorts and consumes the candidates without leaving the SM.
//   * the unsorted candidate keys of the frame (value << idx_bits | pixel index: unique, so "k-th largest" is exact) are
//     taken in chunks of at most kTkCap = 8192, largest first: when more are left than a chunk holds, a radix select
//     (10-bit digits, MSB first, histograms in shared memory) finds the key T with exactly kTkCap keys in [T, upper);
//   * the chunk is gathered into shared memory, sorted with cub::BlockRadixSort (1024 threads x 8 keys, only the
//     significant bits) and handed to warp 0 for the greedy pass; the next chunk is only needed when fewer than
//     max_corners points were accepted and candidates above the quality threshold remain (rare: 0.01 * max cuts the
//     list to ~4.5 k keys at working height 360, ~16 k at 1080).
// Two shapes: 1024 threads x 8 keys (one CTA per SM: a lone frame in streaming wants every thread) and 512 threads x 8
// keys (chunks of 4096; two CTAs per SM when the cell grid leaves room, so a batch of 256 frames is ONE wave over 148 SMs
// instead of two).
template <int kTkThreads, int kTkItems>
struct TkShape {
    static constexpr int kCap = kTkThreads * kTkItems;
    typedef cub::BlockRadixSort<unsigned long long, kTkThreads, kTkItems> Sort;
    union Scratch {
        typename Sort::TempStorage sort;
        unsigned long long keys[kCap];
    };
};

template <int kTkThreads, int kTkItems, int kMinBlocks>
__global__ void __launch_bounds__(kTkThreads, kMinBlocks)
topk_greedy_kernel(const unsigned long long* __restrict__ keys_all, const int* __restrict__ seg_begin,
                   int* __restrict__ seg_end, unsigned int* __restrict__ maxbits, double quality, int idx_bits, int cap,
                   int w, int min_distance, int cell, int grid_w, int grid_h, int max_corners,
                   float2* __restrict__ pts, int* __restrict__ counts) {
    extern __shared__ __align__(16) unsigned char tk_smem[];
    typedef TkShape<kTkThreads, kTkItems> Shape;
    typedef typename Shape::Scratch TkScratch;
    typedef typename Shape::Sort TkSort;
    constexpr int kTkCap = Shape::kCap;
    TkScratch& S = *reinterpret_cast<TkScratch*>(tk_smem);
    unsigned short* gfr = reinterpret_cast<unsigned short*>(tk_smem + sizeof(TkScratch));
    __shared__ unsigned hist[1024];
    __shared__ int bxy[32];
    __shared__ int s_cnt, s_accepted, s_more, s_digit, s_k;
    const int frame = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31;
    const unsigned long long* keys = keys_all + seg_begin[frame];
    const int n = min(seg_end[frame] - seg_begin[frame], cap);
    const int ncells = grid_w * grid_h;
    {
        uint2* g2 = reinterpret_cast<uint2*>(gfr);
        for (int i = tid; i < ncells; i += kTkThreads) g2[i] = make_uint2(0xffffffffu, 0xffffffffu);
    }
    if (tid == 0) { s_accepted = 0; s_more = 1; }
    const float thr = (float)((double)__uint_as_float(maxbits[frame]) * quality);       // cv::threshold takes float(thresh)
    const int key_bits = 31 + idx_bits;
    unsigned long long upper = ~0ull;                  // keys not yet consumed are < upper
    int remaining = n;
    __syncthreads();
    while (remaining > 0) {
        // ---- threshold of this chunk: the kTkCap-th largest key below `upper` (0: take everything that is left)
        unsigned long long T = 0ull;
        if (remaining > kTkCap) {
            unsigned long long prefix = 0ull, pmask = 0ull;
            if (tid == 0) s_k = kTkCap;
            for (int top = key_bits; top > 0; top -= 10) {
                const int shift = top > 10 ? top - 10 : 0;
                const unsigned dmask = (1u << (top - shift)) - 1u;
                for (int i = tid; i < 1024; i += kTkThreads) hist[i] = 0u;
                __syncthreads();
                for (int i0 = tid; i0 < n; i0 += 4 * kTkThreads) {         // 4 loads in flight per thread
                    unsigned long long kk[4];
#pragma unroll
                    for (int u = 0; u < 4; ++u) kk[u] = i0 + u * kTkThreads < n ? keys[i0 + u * kTkThreads] : ~0ull;
#pragma unroll
                    for (int u = 0; u < 4; ++u)
                        if (kk[u] < upper && (kk[u] & pmask) == prefix) atomicAdd(&hist[(unsigned)(kk[u] >> shift) & dmask], 1u);
                }
                __syncthreads();
                if (tid < 32) {
                    // lane l owns digits [32 l, 32 l + 32); find the digit where the count from the top reaches k
                    unsigned sum = 0;
                    for (int d = 0; d < 32; ++d) sum += hist[lane * 32 + d];
                    unsigned above = 0;                // keys in digits owned by higher lanes
                    for (int o = 1; o < 32; ++o) {
                        const unsigned v = __shfl_down_sync(0xffffffffu, sum, o);
                        if (lane + o < 32) above += v;
                    }
                    const unsigned k = (unsigned)s_k;
                    if (above < k && above + sum >= k) {
                        unsigned cum = above;
                        for (int d = 31; d >= 0; --d) {
                            const unsigned c = hist[lane * 32 + d];
                            if (cum + c >= k) { s_digit = lane * 32 + d; s_k = (int)(k - cum); break; }
                            cum += c;
                        }
                    }
                }
                __syncthreads();
                prefix |= (unsigned long long)(unsigned)s_digit << shift;
                pmask |= (unsigned long long)dmask << shift;
                __syncthreads();
            }
            T = prefix;
        }
        // ---- gather the chunk [T, upper) into shared memory, sort it (descending), hand it to warp 0
        if (tid == 0) s_cnt = 0;
        __syncthreads();
        for (int i0 = tid; i0 < n; i0 += 4 * kTkThreads) {
            unsigned long long kk[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) kk[u] = i0 + u * kTkThreads < n ? keys[i0 + u * kTkThreads] : ~0ull;
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (kk[u] >= T && kk[u] < upper) S.keys[atomicAdd(&s_cnt, 1)] = kk[u];
        }
        __syncthreads();
        const int m = s_cnt;
        unsigned long long mine[kTkItems];
#pragma unroll
        for (int i = 0; i < kTkItems; ++i) mine[i] = tid * kTkItems + i < m ? S.keys[tid * kTkItems + i] : 0ull;
        __syncthreads();
        TkSort(S.sort).SortDescending(mine, 0, key_bits);
        __syncthreads();
#pragma unroll
        for (int i = 0; i < kTkItems; ++i) S.keys[tid * kTkItems + i] = mine[i];
        __syncthreads();
        if (tid < 32) {
            int accepted = s_accepted;
            const bool more = greedy_warp(S.keys, m, idx_bits, thr, w, min_distance, cell, grid_w, grid_h, gfr, bxy, max_corners,
                                          pts + (size_t)frame * kMaxCorners, accepted);
            if (lane == 0) { s_accepted = accepted; s_more = (more && accepted < max_corners) ? 1 : 0; }
        }
        __syncthreads();
        remaining -= m;
        upper = T;
        if (!s_more || T == 0ull) break;
    }
    if (tid == 0) {
        counts[frame] = min(s_accepted, max_corners);
        // leave the per-frame counters ready for the next launch (saves a reset kernel per call)
        maxbits[frame] = 0u;
        seg_end[frame] = seg_begin[frame];
    }
}

}  // namespace

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

size_t gftt_workspace_bytes(int w, int h, int min_distance, int max_frames, GfttWorkspace* L) {
    GfttWorkspace ws{};
    ws.max_frames = max_frames;
    ws.cap = (int)align_up((size_t)w * h / 4 + 1024, 256);
    ws.cell = min_distance >= 1 ? min_distance : 1;
    ws.grid_w = (w + ws.cell - 1) / ws.cell;
    ws.grid_h = (h + ws.cell - 1) / ws.cell;
    ws.ncells = ws.grid_w * ws.grid_h;
    ws.grid_in_smem = (size_t)ws.ncells * kCellCap * sizeof(unsigned short) <= (size_t)kGreedySmemMax ? 1 : 0;
    size_t temp = 0;
    cub::DeviceSegmentedRadixSort::SortKeysDescending(
        nullptr, temp, (const unsigned long long*)nullptr, (unsigned long long*)nullptr,
        (int)((size_t)ws.cap * max_frames), max_frames, (const int*)nullptr, (const int*)nullptr, 0, 64);
    ws.cub_temp_bytes = temp;
    ws.idx_bits = 1;
    while (((size_t)1 << ws.idx_bits) < (size_t)w * h) ++ws.idx_bits;
    ws.counters_ready = 0;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
    // offsets are stored in the pointer fields and rebased by gftt_bind_workspace
    ws.eig = (float*)take((size_t)w * h * sizeof(float));            // one frame: parity tap only
    ws.maxbits = (unsigned int*)take((size_t)max_frames * sizeof(unsigned int));
    ws.keys = (unsigned long long*)take((size_t)max_frames * ws.cap * sizeof(unsigned long long));
    ws.keys_alt = (unsigned long long*)take((size_t)max_frames * ws.cap * sizeof(unsigned long long));
    ws.seg_begin = (int*)take((size_t)max_frames * sizeof(int));
    ws.seg_end = (int*)take((size_t)max_frames * sizeof(int));
    ws.grid = (unsigned short*)take(ws.grid_in_smem ? 16 : (size_t)max_frames * ws.ncells * kCellCap * sizeof(unsigned short));
    ws.cub_temp = (void*)take(temp);
    *L = ws;
    return off;
}

void gftt_bind_workspace(void* base, GfttWorkspace* ws) {
    char* b = (char*)base;
    ws->eig = (float*)(b + (size_t)ws->eig);
    ws->maxbits = (unsigned int*)(b + (size_t)ws->maxbits);
    ws->keys = (unsigned long long*)(b + (size_t)ws->keys);
    ws->keys_alt = (unsigned long long*)(b + (size_t)ws->keys_alt);
    ws->seg_begin = (int*)(b + (size_t)ws->seg_begin);
    ws->seg_end = (int*)(b + (size_t)ws->seg_end);
    ws->grid = (unsigned short*)(b + (size_t)ws->grid);
    ws->cub_temp = (void*)(b + (size_t)ws->cub_temp);
}

void launch_gftt(const uint8_t* gray, size_t gray_frame_stride, int w, int h, int nframes,
                 double quality, int min_distance, int max_corners, GfttWorkspace& ws,
                 float2* pts, int* counts, float* eig_out, cudaStream_t st) {
    if (nframes <= 0) return;
    if (max_corners > kMaxCorners) max_corners = kMaxCorners;
    const size_t grid_bytes = (size_t)ws.ncells * kCellCap * sizeof(unsigned short);
    typedef TkShape<1024, 8> Big;
    typedef TkShape<512, 8> Small;
    const size_t fused_smem = sizeof(Big::Scratch) + grid_bytes;
    const size_t small_smem = sizeof(Small::Scratch) + grid_bytes;
    // the unfused schedule (clamp, cub sort, greedy_kernel) serves cell grids that do not fit beside the top-k scratch:
    // small working heights, where min_distance is 1 and a cell is one pixel
    const bool fused = fused_smem <= (size_t)220 * 1024;
    // batches larger than one wave of single-CTA SMs: the half-size shape when two of its CTAs fit an SM
    // (227 KB shared memory per SM, 1 KB reserved per CTA, + the static histogram)
    static PerDeviceOnce once;
    once.run([] {
        cudaFuncSetAttribute(greedy_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kGreedySmemMax);
        cudaFuncSetAttribute(topk_greedy_kernel<1024, 8, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024);
        cudaFuncSetAttribute(topk_greedy_kernel<512, 8, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 110 * 1024);
    });
    const int num_sms = device_sm_count();
    const bool use_small = fused && nframes > num_sms && small_smem <= (size_t)108 * 1024;
    const int key_bits = 31 + ws.idx_bits;
    // the fused kernel leaves the per-frame counters reset behind it
    if (!(fused && ws.counters_ready && nframes == 1)) {
        count_launch(1);
        gftt_reset_kernel<<<(nframes + 127) / 128, 128, 0, st>>>(ws.maxbits, ws.seg_begin, ws.seg_end, ws.cap, nframes);
    }
    ws.counters_ready = fused ? 1 : 0;
    {
        // rows per warp: long segments amortise the 4 halo rows; a few frames alone (streaming) want more, shorter
        // warps instead (latency)
        const int seg_h = nframes >= 8 ? kSegH : 15;
        const int nstrips = (w + kStripW - 1) / kStripW, nsegs = (h + seg_h - 1) / seg_h;
        dim3 grid((nstrips * nsegs + kEigWarps - 1) / kEigWarps, nframes);
        count_launch(1);
        eig_kernel<<<grid, 32 * kEigWarps, 0, st>>>(gray, gray_frame_stride, w, h, nstrips, nsegs, seg_h, ws.idx_bits, eig_out, ws.maxbits,
                                                    ws.keys, ws.seg_end, ws.cap, quality, kEigPrefetchRows);
    }
    if (fused) {
        count_launch(1);
        if (use_small)
            topk_greedy_kernel<512, 8, 2><<<nframes, 512, small_smem, st>>>(ws.keys, ws.seg_begin, ws.seg_end, ws.maxbits, quality,
                                                                           ws.idx_bits, ws.cap, w, min_distance, ws.cell, ws.grid_w,
                                                                           ws.grid_h, max_corners, pts, counts);
        else
            topk_greedy_kernel<1024, 8, 1><<<nframes, 1024, fused_smem, st>>>(ws.keys, ws.seg_begin, ws.seg_end, ws.maxbits, quality,
                                                                             ws.idx_bits, ws.cap, w, min_distance, ws.cell, ws.grid_w,
                                                                             ws.grid_h, max_corners, pts, counts);
        return;
    }
    // unfused schedule: clamp, cub radix sort (its passes are not counted as launches of ours), greedy
    count_launch(2);
    clamp_segments_kernel<<<(nframes + 127) / 128, 128, 0, st>>>(ws.seg_end, ws.cap, nframes);
    size_t temp = ws.cub_temp_bytes;
    cub::DeviceSegmentedRadixSort::SortKeysDescending(
        ws.cub_temp, temp, (const unsigned long long*)ws.keys, ws.keys_alt, (int)((size_t)ws.cap * nframes),
        nframes, (const int*)ws.seg_begin, (const int*)ws.seg_end, 0, key_bits, st);
    const size_t smem = ws.grid_in_smem ? grid_bytes : 0;
    greedy_kernel<<<nframes, kGreedyThreads, smem, st>>>(ws.keys_alt, ws.seg_begin, ws.seg_end, ws.maxbits, quality, ws.idx_bits, w,
                                                         min_distance, ws.cell, ws.grid_w, ws.grid_h, ws.grid, ws.grid_in_smem,
                                                         max_corners, pts, counts);
}

}  // namespace vstabk
