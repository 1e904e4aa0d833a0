// K7: fused output warp
//   cv::warpPerspective(presentation_image, warped, H_stabilize_scaled, frame.size(),
//                       INTER_LINEAR, BORDER_CONSTANT, 0.5*mean)      /root/reference/src/stabilizer.cpp:1309-1313
// Bit-exact restatement of OpenCV's fixed-point path (SURVEY A.11): inverse map in f64,
// (X,Y)*32/W rounded half-even to Q5, 2x2 taps with Q15 weights
//   w = {(32-ay)(32-ax), (32-ay)ax, ay(32-ax), ay ax} * 32     (== OpenCV's int16 table; the one
//   saturated entry (0,0) -> {32767,1,0,0} yields the same pixel, see DESIGN.md),
// out = (sum + 16384) >> 15, taps outside the source take the constant border colour.
// HBM-bound by design: reads 3WH, writes 3WH per frame.
//
// One 128 x 32 destination tile at a time.  Every H the stabilizer produces is affine (SURVEY B.8),
// so the source footprint of a tile is a small parallelogram: its bounding box is staged in shared
// memory and the taps are read from there as aligned 32-bit words + funnel shifts.  All four Q15
// weights carry the factor 32, so out = (sum_i p_i w_i / 32 + 512) >> 10 with 11-bit weights: per
// channel the four taps sit in one word and the sum is two dp2a (16-bit weights x 8-bit pixels).
//   * interior tiles (the unclamped footprint lies inside the image): branch-free path, no per-tap tests;
//   * tiles touching the image border, non-affine H, footprints larger than a stage: per-pixel path with
//     border substitution (generic_pixel).
// One CTA per tile; the box is filled with 16-byte cp.async copies by the CTA itself.
#include <cstring>
#include "kernels.h"

namespace vstabk {
namespace {

constexpr int TW = 128, TH = 32;               // destination tile
constexpr int NTX = 32, NTY = 8;               // threads: 4 px per thread in x, TH/NTY rows per thread
constexpr int kStageBytes = 40 * 1024;         // staged source box
constexpr int kStageStride = kStageBytes + 128; // + slack for the 3-word tap loads of the last pixel

struct Taps6 { unsigned lo, hi; };  // bytes A..A+7 (6 used: two BGR pixels)

VSTAB_D Taps6 load6(const uint8_t* row, int byte_off) {
    const int al = byte_off & ~3;
    const int sh = (byte_off & 3) * 8;
    const unsigned* p = reinterpret_cast<const unsigned*>(row + al);
    const unsigned w0 = __ldg(p), w1 = __ldg(p + 1), w2 = __ldg(p + 2);
    Taps6 t;
    t.lo = __funnelshift_r(w0, w1, sh);
    t.hi = __funnelshift_r(w1, w2, sh);
    return t;
}

VSTAB_D int byte_of(const Taps6& t, int i) {   // i in 0..5
    return i < 4 ? (int)((t.lo >> (8 * i)) & 0xffu) : (int)((t.hi >> (8 * (i - 4))) & 0xffu);
}

// Generic pixel: taps from global memory, border substitution (OpenCV remap semantics incl. the
// int16 saturation of the integer coordinates).  Returns packed B | G<<8 | R<<16.
__device__ __noinline__ unsigned generic_pixel(const uint8_t* __restrict__ src, size_t pitch, int w, int h, bool al_ok,
                                               int iX, int iY, const int* sB) {
    int sx = iX >> 5, sy = iY >> 5;
    // all four taps outside the source: the weights sum to 2^15, so the pixel is the border colour
    if (sx < -1 || sx >= w || sy < -1 || sy >= h) return (unsigned)sB[0] | ((unsigned)sB[1] << 8) | ((unsigned)sB[2] << 16);
    const int ax = iX & 31, ay = iY & 31;
    sx = max(-32768, min(32767, sx));      // remap stores int16 coordinates
    sy = max(-32768, min(32767, sy));
    const int w00 = (32 - ay) * (32 - ax) * 32, w01 = (32 - ay) * ax * 32;
    const int w10 = ay * (32 - ax) * 32, w11 = ay * ax * 32;
    int p00[3], p01[3], p10[3], p11[3];
    const bool fast = al_ok && sx >= 0 && sy >= 0 && sy + 1 < h && 3 * sx + 14 <= 3 * w;
    if (fast) {
        const uint8_t* r0 = src + (size_t)sy * pitch;
        const Taps6 a = load6(r0, 3 * sx);
        const Taps6 b = load6(r0 + pitch, 3 * sx);
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            p00[c] = byte_of(a, c); p01[c] = byte_of(a, 3 + c);
            p10[c] = byte_of(b, c); p11[c] = byte_of(b, 3 + c);
        }
    } else {
        const bool y0in = sy >= 0 && sy < h, y1in = sy + 1 >= 0 && sy + 1 < h;
        const bool x0in = sx >= 0 && sx < w, x1in = sx + 1 >= 0 && sx + 1 < w;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            p00[c] = (y0in && x0in) ? (int)__ldg(src + (size_t)sy * pitch + 3 * sx + c) : sB[c];
            p01[c] = (y0in && x1in) ? (int)__ldg(src + (size_t)sy * pitch + 3 * (sx + 1) + c) : sB[c];
            p10[c] = (y1in && x0in) ? (int)__ldg(src + (size_t)(sy + 1) * pitch + 3 * sx + c) : sB[c];
            p11[c] = (y1in && x1in) ? (int)__ldg(src + (size_t)(sy + 1) * pitch + 3 * (sx + 1) + c) : sB[c];
        }
    }
    unsigned res = 0;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const int v = (p00[c] * w00 + p01[c] * w01 + p10[c] * w10 + p11[c] * w11 + 16384) >> 15;
        res |= (unsigned)min(255, max(0, v)) << (8 * c);
    }
    return res;
}

constexpr int kSP = 512;                       // row stride of the staged box (bytes)

// Bilinear blend of one pixel from the staged box: byte offset `o` of its top-left tap, Q5 fractions ax, ay.
// Each row's 6 tap bytes (two BGR pixels) come from three aligned words + two funnel shifts; the row stride is a
// multiple of 4, so both rows share the word alignment and the shift amount.  Returns acc_b, acc_g, acc_r with the
// pixel value in bits 10..17.
VSTAB_D void staged_taps(const uint8_t* __restrict__ sm, int o, unsigned ax, unsigned ay, unsigned& ab, unsigned& ag, unsigned& ar) {
    const unsigned* p = reinterpret_cast<const unsigned*>(sm + (o & ~3));
    const unsigned a0 = p[0], a1 = p[1], a2 = p[2];
    const unsigned b0 = p[kSP / 4], b1 = p[kSP / 4 + 1], b2 = p[kSP / 4 + 2];
    const unsigned sh = (unsigned)o << 3;                        // the shifter uses sh & 31 = 8 * (o & 3)
    const unsigned loA = __funnelshift_r(a0, a1, sh), hiA = __funnelshift_r(a1, a2, sh);   // B0 G0 R0 B1 | G1 R1 . .
    const unsigned loB = __funnelshift_r(b0, b1, sh), hiB = __funnelshift_r(b1, b2, sh);
    // per channel the four taps in one word {p00, p01, p10, p11}
    const unsigned tA = __byte_perm(loA, hiA, 0x5241);          // G0 G1 R0 R1 of row A
    const unsigned tB = __byte_perm(loB, hiB, 0x5241);
    const unsigned WB = __byte_perm(loA, loB, 0x7430);
    const unsigned WG = __byte_perm(tA, tB, 0x5410);
    const unsigned WR = __byte_perm(tA, tB, 0x7632);
    // 16-bit weight pairs {w00, w01} = (32-ay) * {32-ax, ax}, {w10, w11} = ay * {32-ax, ax}   (<= 1024: no carries)
    const unsigned wxp = ax * 0xffffu + 32u;                    // (32-ax) | ax << 16
    const unsigned w23 = ay * wxp, w01 = (wxp << 5) - w23;
    ab = __dp2a_hi(w23, WB, __dp2a_lo(w01, WB, 512u));
    ag = __dp2a_hi(w23, WG, __dp2a_lo(w01, WG, 512u));
    ar = __dp2a_hi(w23, WR, __dp2a_lo(w01, WR, 512u));
}
// B | G << 8 | R << 16 from the accumulators (value in bits 10..17 of each)
VSTAB_D unsigned pack_bgr(unsigned ab, unsigned ag, unsigned ar) {
    return __byte_perm(__byte_perm(ab >> 10, ag >> 2, 0x1150), ar << 6, 0x3610);
}
VSTAB_D unsigned staged_pixel(const uint8_t* __restrict__ sm, int o, unsigned ax, unsigned ay) {
    unsigned ab, ag, ar;
    staged_taps(sm, o, ax, ay, ab, ag, ar);
    return pack_bgr(ab, ag, ar);
}

// staged box: x in [fx0, fx0+fxn], y in [fy0, fy0+fyn]; rows of `nb` bytes (from byte b0 of the source row) at a
// stride of SP = kSP = 512 bytes (0: nothing staged): a multiple of 128, so that a lane whose taps sit one source
// row lower hits the same banks (lanes are 3 words apart along a row: conflict-free).  `inside`: the unclamped footprint lies inside the
// image, i.e. every tap of every pixel of the tile is in the box -> the branch-free path.
struct TileBox { int fx0, fxn, fy0, fyn, b0, SP, nb, inside; };

// Everything the CTA needs to know about its destination tile.
struct TileInfo {
    double M[9];
    const uint8_t* src;
    TileBox box;
    int border[3];
    int oi, tx0, ty0, slot;
};

// Source bounding box of the destination tile at (tx0, ty0) under the inverse map M, when M is affine and the box
// fits a stage; otherwise the empty box.  The box is clipped to the image (the ld.global fill must not leave it).
VSTAB_D TileBox tile_box(const double* M, const uint8_t* src, size_t pitch, int w, int h, int tx0, int ty0) {
    TileBox bx{0, 0, 0, 0, 0, 0, 0, 0};                                      // empty: nothing staged, no pixel is "inside"
    const bool al_ok = ((pitch & 15) == 0) && ((reinterpret_cast<uintptr_t>(src) & 15) == 0);
    if (M[6] == 0.0 && M[7] == 0.0 && M[8] != 0.0 && al_ok) {
        // the tile's source footprint is a parallelogram whose extremes are at the tile corners
        const int tx1 = min(tx0 + TW, w) - 1, ty1 = min(ty0 + TH, h) - 1;
        const double wd = 1.0 / M[8];
        double xmn = 1e300, xmx = -1e300, ymn = 1e300, ymx = -1e300;
        for (int c = 0; c < 4; ++c) {
            const double cx = (c & 1) ? (double)tx1 : (double)tx0, cy = (c & 2) ? (double)ty1 : (double)ty0;
            const double X = (M[0] * cx + M[1] * cy + M[2]) * wd, Y = (M[3] * cx + M[4] * cy + M[5]) * wd;
            xmn = fmin(xmn, X); xmx = fmax(xmx, X); ymn = fmin(ymn, Y); ymx = fmax(ymx, Y);
        }
        if (xmx > -4.0 && ymx > -4.0 && xmn < (double)w + 4.0 && ymn < (double)h + 4.0) {
            // a pixel's taps are at floor(iX/32), +1 with iX = rint(32 X): >= floor(X) - 1 and <= floor(X) + 2
            const int ux0 = (int)floor(xmn) - 1, ux1 = (int)floor(xmx) + 2;
            const int uy0 = (int)floor(ymn) - 1, uy1 = (int)floor(ymx) + 2;
            const int inside = (ux0 >= 0 && ux1 <= w - 1 && uy0 >= 0 && uy1 <= h - 1) ? 1 : 0;
            const int fx0 = max(0, ux0), fx1 = min(w - 1, ux1);
            const int fy0 = max(0, uy0), fy1 = min(h - 1, uy1);
            const int b0 = (3 * fx0) & ~15;
            const int b1 = min((int)pitch, (3 * (fx1 + 1) + 15) & ~15);
            const int nb = b1 - b0;
            if (fx1 > fx0 && fy1 > fy0 && nb <= kSP && kSP * (fy1 - fy0 + 1) <= kStageBytes)
                bx = TileBox{fx0, fx1 - fx0, fy0, fy1 - fy0, b0, kSP, nb, inside};
        }
    }
    return bx;
}

// Per-frame output checksum (offline jobs whose output is never downloaded, e.g. BASELINE config 5): over the tight
// rows of the frame, cut into 12-byte groups (4 pixels, the last group zero-padded) read as three little-endian words,
//   checksum = sum_y sum_g (y + 1) (g + 1) (w0 + 3 w1 + 5 w2)   mod 2^64
// (order-free, so every tiling and every shard split gives the same value; numpy twin: vstab_b200.frame_checksum).
struct RowSums { unsigned long long a = 0; };   // sum over the thread's rows of (y + 1) (w0 + 3 w1 + 5 w2)

template <bool kCheck>
VSTAB_D void store4(uint8_t* __restrict__ o, const unsigned* px, bool vec, int n, int y, RowSums& cs) {
    const unsigned w0 = __byte_perm(px[0], px[1], 0x4210), w1 = __byte_perm(px[1], px[2], 0x5421), w2 = __byte_perm(px[2], px[3], 0x6542);
    if (vec) {
        unsigned* o32 = reinterpret_cast<unsigned*>(o);
        o32[0] = w0; o32[1] = w1; o32[2] = w2;
        if (kCheck) cs.a += ((unsigned long long)w0 + 3ull * w1 + 5ull * w2) * (unsigned)(y + 1);
    } else {
        for (int k = 0; k < n; ++k) {
            o[3 * k] = (uint8_t)(px[k] & 0xff); o[3 * k + 1] = (uint8_t)((px[k] >> 8) & 0xff); o[3 * k + 2] = (uint8_t)(px[k] >> 16);
        }
        if (kCheck) {
            // bytes beyond pixel n - 1 count as zero
            const unsigned long long lo = (unsigned long long)w0 | ((unsigned long long)w1 << 32);
            const int nb = 3 * n;                                         // valid bytes of the 12
            const unsigned long long mlo = nb >= 8 ? ~0ull : ((1ull << (8 * nb)) - 1ull);
            const unsigned m2 = nb >= 12 ? ~0u : (nb <= 8 ? 0u : ((1u << (8 * (nb - 8))) - 1u));
            const unsigned v0 = (unsigned)(lo & mlo), v1 = (unsigned)((lo & mlo) >> 32), v2 = w2 & m2;
            cs.a += ((unsigned long long)v0 + 3ull * v1 + 5ull * v2) * (unsigned)(y + 1);
        }
    }
}

// The 128 x 32 destination tile at (tx0, ty0): thread (tx, ty) of the 32 x 8 thread tile produces
// 4 consecutive pixels on each of the rows ty, ty+8, ty+16, ty+24.
// Interior tile: every tap is in the staged box, M is affine.
template <bool kCheck>
VSTAB_D void compute_tile_inside(const uint8_t* __restrict__ sm, const TileBox box, const double* M, int w, int h,
                                 uint8_t* __restrict__ dst, size_t out_pitch, int tx0, int ty0, int tx, int ty, RowSums& cs) {
    const int x0 = tx0 + tx * 4;
    if (x0 >= w) return;
    const double M0 = M[0], M1 = M[1], M2 = M[2], M3 = M[3], M4 = M[4], M5 = M[5];
    const double wdiv = __ddiv_rn(32.0, M[8]);
    const bool vec = x0 + 4 <= w && (out_pitch & 3) == 0 && ((reinterpret_cast<uintptr_t>(dst) & 3) == 0);
    const int obase = -box.fy0 * kSP - box.b0;
    // OpenCV evaluates per 32-px block: X0 = M0*bx + M1*y + M2, then X0 + M0*x1
    const double bx = (double)(x0 & ~31);
    const double XB = __dmul_rn(M0, bx), YB = __dmul_rn(M3, bx);
    double mx1[4], my1[4];                        // M0*x1, M3*x1 for the 4 pixels of this thread
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const double x1 = (double)((x0 + i) & 31);
        mx1[i] = __dmul_rn(M0, x1);
        my1[i] = __dmul_rn(M3, x1);
    }
    uint8_t* orow = dst + (size_t)(ty0 + ty) * out_pitch + (size_t)x0 * 3;
    const int yend = min(ty0 + TH, h);
#pragma unroll 1
    for (int y = ty0 + ty; y < yend; y += NTY, orow += (size_t)NTY * out_pitch) {
        const double yd = (double)y;
        const double X0 = __dadd_rn(__dadd_rn(XB, __dmul_rn(M1, yd)), M2);
        const double Y0 = __dadd_rn(__dadd_rn(YB, __dmul_rn(M4, yd)), M5);
        unsigned px[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            // saturate_cast<int>(X * 32/W): cvt.rni.s32.f64 saturates like OpenCV's explicit clamp
            const int iX = __double2int_rn(__dmul_rn(__dadd_rn(X0, mx1[i]), wdiv));
            const int iY = __double2int_rn(__dmul_rn(__dadd_rn(Y0, my1[i]), wdiv));
            const int o = (iY >> 5) * kSP + 3 * (iX >> 5) + obase;
            px[i] = staged_pixel(sm, o, iX & 31, iY & 31);
        }
        store4<kCheck>(orow, px, vec, min(4, w - x0), y, cs);
    }
}

// Any tile: per-pixel test against the staged box (may be empty), generic_pixel otherwise.
template <bool kAffine, bool kCheck>
VSTAB_D void compute_tile_border(const uint8_t* __restrict__ sm, const TileBox box, const double* M, const int* border,
                                 const uint8_t* __restrict__ src, size_t pitch, int w, int h,
                                 uint8_t* __restrict__ dst, size_t out_pitch, int tx0, int ty0, int tx, int ty, RowSums& cs) {
    const int x0 = tx0 + tx * 4;
    if (x0 >= w) return;
    const double M0 = M[0], M1 = M[1], M2 = M[2], M3 = M[3], M4 = M[4], M5 = M[5], M6 = M[6], M7 = M[7], M8 = M[8];
    const bool al_ok = ((pitch & 15) == 0) && ((reinterpret_cast<uintptr_t>(src) & 15) == 0);
    const double bx = (double)(x0 & ~31);
    const double wdiv = kAffine ? __ddiv_rn(32.0, M8) : 0.0;
    const bool vec = x0 + 4 <= w && (out_pitch & 3) == 0 && ((reinterpret_cast<uintptr_t>(dst) & 3) == 0);
    const int obase = -box.fy0 * kSP - box.b0;
    // a pixel reads the stage when its taps sx, sx + 1 and sy, sy + 1 all lie in the box
    const int cx0 = max(box.fx0, 0), cxn = box.SP > 0 ? max(min(box.fx0 + box.fxn, w - 1) - cx0, 0) : 0;
    const int cy0 = max(box.fy0, 0), cyn = box.SP > 0 ? max(min(box.fy0 + box.fyn, h - 1) - cy0, 0) : 0;
    const double XB = __dmul_rn(M0, bx), YB = __dmul_rn(M3, bx), WB = __dmul_rn(M6, bx);
    const int yend = min(ty0 + TH, h);
#pragma unroll 1
    for (int y = ty0 + ty; y < yend; y += NTY) {
        const double yd = (double)y;
        const double X0 = __dadd_rn(__dadd_rn(XB, __dmul_rn(M1, yd)), M2);
        const double Y0 = __dadd_rn(__dadd_rn(YB, __dmul_rn(M4, yd)), M5);
        const double W0 = __dadd_rn(__dadd_rn(WB, __dmul_rn(M7, yd)), M8);
        unsigned px[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const double x1 = (double)((x0 + i) & 31);
            const double X = __dadd_rn(X0, __dmul_rn(M0, x1));
            const double Y = __dadd_rn(Y0, __dmul_rn(M3, x1));
            double Wd = wdiv;
            if (!kAffine) {
                const double W = __dadd_rn(W0, __dmul_rn(M6, x1));
                Wd = W != 0.0 ? __ddiv_rn(32.0, W) : 0.0;
            }
            const int iX = __double2int_rn(__dmul_rn(X, Wd)), iY = __double2int_rn(__dmul_rn(Y, Wd));
            const int sx = iX >> 5, sy = iY >> 5;
            if ((unsigned)(sx - cx0) < (unsigned)cxn && (unsigned)(sy - cy0) < (unsigned)cyn)
                px[i] = staged_pixel(sm, sy * kSP + 3 * sx + obase, iX & 31, iY & 31);
            else
                px[i] = generic_pixel(src, pitch, w, h, al_ok, iX, iY, border);
        }
        store4<kCheck>(dst + (size_t)y * out_pitch + (size_t)x0 * 3, px, vec, min(4, w - x0), y, cs);
    }
}

// One destination tile, whichever path it needs.  kCheck: the thread's share of the frame checksum goes to *check
// (one 64-bit atomic per warp).
template <bool kCheck>
VSTAB_D void compute_tile(const uint8_t* __restrict__ sm, const TileBox box, const double* M, const int* border,
                          const uint8_t* __restrict__ src, size_t pitch, int w, int h,
                          uint8_t* __restrict__ dst, size_t out_pitch, int tx0, int ty0, int tx, int ty,
                          unsigned long long* check) {
    RowSums cs;
    if (box.inside)
        compute_tile_inside<kCheck>(sm, box, M, w, h, dst, out_pitch, tx0, ty0, tx, ty, cs);
    else if (M[6] == 0.0 && M[7] == 0.0 && M[8] != 0.0)
        compute_tile_border<true, kCheck>(sm, box, M, border, src, pitch, w, h, dst, out_pitch, tx0, ty0, tx, ty, cs);
    else
        compute_tile_border<false, kCheck>(sm, box, M, border, src, pitch, w, h, dst, out_pitch, tx0, ty0, tx, ty, cs);
    if (kCheck) {
        const unsigned long long g1 = (unsigned long long)((tx0 + tx * 4) >> 2) + 1ull;
        unsigned long long c = (tx0 + tx * 4 < w) ? cs.a * g1 : 0ull;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
        if (tx == 0) atomicAdd(check, c);
    }
}

VSTAB_D void fill_tile_info(TileInfo& I, const WarpParams& P, const uint8_t* frames, size_t frame_stride, long slot_mod) {
#pragma unroll
    for (int i = 0; i < 9; ++i) I.M[i] = P.Minv[i];
    I.border[0] = P.border[0]; I.border[1] = P.border[1]; I.border[2] = P.border[2];
    I.slot = (int)(slot_mod > 0 ? (P.src_slot % slot_mod) : P.src_slot);
    I.src = frames + (size_t)I.slot * frame_stride;
}

template <bool kCheck>
__global__ void __launch_bounds__(NTX * NTY, 4)
warp_tile_kernel(const uint8_t* __restrict__ frames, size_t pitch, size_t frame_stride, long slot_mod,
                 const WarpParams* __restrict__ wps, int w, int h,
                 uint8_t* __restrict__ out, size_t out_pitch, size_t out_frame_stride, unsigned long long* __restrict__ check) {
    __shared__ __align__(128) uint4 stage[kStageStride / 16];
    __shared__ TileInfo I;
    const int oi = blockIdx.z;
    const int tid = threadIdx.y * NTX + threadIdx.x;
    const int tx0 = blockIdx.x * TW, ty0 = blockIdx.y * TH;
    if (tid == 0) {
        fill_tile_info(I, wps[oi], frames, frame_stride, slot_mod);
        I.box = tile_box(I.M, I.src, pitch, w, h, tx0, ty0);
    }
    __syncthreads();
    const TileBox box = I.box;
    if (box.SP > 0) {
        // nb <= 512: one 16-byte chunk per lane and row
        const int vpr = box.nb >> 4;
        // asynchronous 16-byte copies (LDGSTS): every row of the box is in flight at once, no registers involved
        if ((int)threadIdx.x < vpr) {
            const uint8_t* g = I.src + (size_t)box.fy0 * pitch + box.b0 + (size_t)threadIdx.x * 16;
            const unsigned d = (unsigned)__cvta_generic_to_shared(stage) + threadIdx.x * 16;
            for (int r = threadIdx.y; r <= box.fyn; r += NTY)
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d + r * kSP), "l"(g + (size_t)r * pitch) : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        asm volatile("cp.async.wait_group 0;" ::: "memory");
    }
    __syncthreads();
    uint8_t* dst = out + (size_t)oi * out_frame_stride;
    compute_tile<kCheck>(reinterpret_cast<const uint8_t*>(stage), box, I.M, I.border, I.src, pitch, w, h, dst, out_pitch, tx0, ty0,
                         threadIdx.x, threadIdx.y, kCheck ? check + oi : nullptr);
}

}  // namespace

void launch_warp(const uint8_t* frames, size_t pitch, size_t frame_stride, long slot_mod,
                 const WarpParams* wp, int nout, int w, int h,
                 uint8_t* out, size_t out_pitch, size_t out_frame_stride, cudaStream_t st, unsigned long long* check) {
    if (nout <= 0) return;
    count_launch(1);
    dim3 grid((w + TW - 1) / TW, (h + TH - 1) / TH, nout);
    if (check)
        warp_tile_kernel<true><<<grid, dim3(NTX, NTY), 0, st>>>(frames, pitch, frame_stride, slot_mod, wp, w, h, out, out_pitch,
                                                                out_frame_stride, check);
    else
        warp_tile_kernel<false><<<grid, dim3(NTX, NTY), 0, st>>>(frames, pitch, frame_stride, slot_mod, wp, w, h, out, out_pitch,
                                                                 out_frame_stride, nullptr);
}

}  // namespace vstabk
