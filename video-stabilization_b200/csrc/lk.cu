// K4: sparse pyramidal Lucas-Kanade, one warp per feature
//   == cv::calcOpticalFlowPyrLK(prevGray, gray, prevPts, ..., Size(21,21), 3,
//                               {COUNT+EPS, 50, 0.01}, 0, 1e-4)
// (/root/reference/src/stabilizer.cpp:170-209).  Control flow, fixed-point formats and
// float operation order follow OpenCV's LKTrackerInvoker (SURVEY A.4): Q14 bilinear
// weights, Q5 intensity patches, Scharr derivatives (zero outside the image, intensity
// reflect-101 padded), float 2x2 normal equations, eps^2 = 1e-4, oscillation damping.
//
// BIT-EXACT with OpenCV 4.x (SSE2/universal-intrinsics build), including the float rounding of the
// 441-term sums.  OpenCV accumulates each sum in FIVE float chains, row-major over the window:
//   chain k = 0..3 : the four lanes of a v_float32x4 over the columns x < 16 with x % 4 == k
//                    (A sums: one term per pixel, product then add; b sums: the int32 pair
//                    P(y,x) + P(y,x+4) of an 8-column block converted to float, then added),
//   chain 4        : the scalar tail over the columns 16..20 (float(int product) added one by one),
//   result         = chain4 + ((chain0 + chain2) + (chain1 + chain3))         (v_reduce_sum, SSE order).
// Every term is an integer, so a chain is exact -- and therefore order-free -- as long as the absolute
// values of its terms sum to less than 2^24.  The kernel keeps OpenCV's value in three tiers:
//   tier 0: the bound holds for the whole window          -> one exact warp sum,
//   tier 1: the bound holds for every chain                -> five exact chain sums, OpenCV's four adds,
//   tier 2: otherwise the terms go through shared memory in chain order and 10 (b) / 15 (A) lanes
//           replay the sequential float additions.
// The A sums (once per level) always take the replay; the b sums (every iteration) take the tiers.
//
// The 21x21 template (I, Ix, Iy) of a level lives in registers: the window is cut into 63 vertical
// strips of 7 pixels (3 strip rows x 21 columns), two per lane, both of the same chain: lanes 0..23
// own the column pair (x, x + 4) of an 8-column block (x = 0..3, 8..11) in strip row lane / 8 -- the
// pair whose products OpenCV adds as integers -- and lanes 24..31 the 15 strips of the columns 16..20.
// Every level of a frame's pyramid block has the same row pitch, so with the pitch as a template
// argument the 7 taps of a strip are ONE pointer + immediate offsets.  Intensities come from the padded
// u8 level (reflect-101 border) and derivatives from the padded Scharr level (zero border) that K2
// prepares, so no tap ever needs border logic; both are tiny and L1/L2-resident.
#include "kernels.h"

namespace vstabk {
namespace {

constexpr int kPix = kLkWin * kLkWin;  // 441

// dp2a with signed 16-bit weights and unsigned 8-bit pixels (w11 = 2^14 - w00 - w01 - w10 can be -1):
// d = c + a.s16[0] * b.u8[2*hi] + a.s16[1] * b.u8[2*hi+1]
VSTAB_D int dp2a_lo_su(unsigned a, unsigned b, int c) {
    int d;
    asm("dp2a.lo.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
VSTAB_D int dp2a_hi_su(unsigned a, unsigned b, int c) {
    int d;
    asm("dp2a.hi.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
// keep a computed pointer in registers (ptxas otherwise rematerialises the 64-bit base arithmetic at every tap)
VSTAB_D const unsigned* pin(const unsigned* p) {
    asm volatile("" : "+l"(p));
    return p;
}
VSTAB_D unsigned pack_w(int lo, int hi) { return ((unsigned)lo & 0xffffu) | ((unsigned)hi << 16); }

// exact int -> float for |v| < 2^22 without the conversion pipe: 1.5 * 2^23 + v is representable
VSTAB_D float small_int_to_float(int v) { return __fsub_rn(__int_as_float(0x4B400000 + v), 12582912.f); }

// OpenCV's final reduction of the five chain sums (v_reduce_sum of the SSE build: (q0 + q2) + (q1 + q3), then the scalar tail)
VSTAB_D float combine_chains(float c0, float c1, float c2, float c3, float c4) {
    return __fadd_rn(c4, __fadd_rn(__fadd_rn(c0, c2), __fadd_rn(c1, c3)));
}


// Shared-memory geometry of a lane, recomputed where it is used (a handful of integer instructions) instead of
// being held in registers across the whole kernel: `l` is an opaque copy of the lane index, so nothing is hoisted.
struct LaneGeo { int oa, ob, sa, ta, tb, sb; };
VSTAB_D LaneGeo lane_geo(int l) {
    asm volatile("" : "+r"(l));
    LaneGeo g;
    if (l < 24) {
        const int r = l & 7, q = l >> 3, ch = r & 3;
        g.oa = 84 * ch + 28 * q + (r >> 2) * 2; g.ob = g.oa + 1; g.sa = 4;      // column c0 = ch + 8 (r >> 2): c0 >> 2 = 2 (r >> 2)
        g.ta = g.tb = 44 * ch + 14 * q + (r >> 2); g.sb = 2;
    } else {
        const int i0 = 2 * (l - 24), i1 = i0 + 1 < 15 ? i0 + 1 : 14;
        g.oa = 336 + 7 * i0 - 6 * (i0 % 5) + 0 * i1; g.ob = 0; g.sa = 5;       // 35 (i / 5) + i % 5 = 7 i - 6 (i % 5)
        g.ob = 336 + 7 * i1 - 6 * (i1 % 5);
        g.ta = g.oa - 160; g.tb = g.ob - 160; g.sb = 5;                          // 176 + ... = 336 + ... - 160
    }
    return g;
}
// replay lanes: lane = 5 * sum + chain (A: sums A11, A12, A22 on lanes 0..14; b: b1, b2 on lanes 0..9)
VSTAB_D void replay_geo(int l, int& rs, int& rc) {
    asm volatile("" : "+r"(l));
    rs = l / 5; rc = l - 5 * rs;
}

constexpr int kStripLen = 7;
// shared memory per warp, in floats.  A planes (Ix, Iy in chain order): chains 0..3 at 84 c (84 terms: row * 4 + x / 4), chain 4
// at 336 (105 terms: row * 5 + x - 16), 3 zero pads.  b planes (terms of b1, b2 in chain order) alias them: chains 0..3 at 44 c
// (42 pair terms: row * 2 + block, 2 zero pads), chain 4 at 176 (105 terms, 3 zero pads).
constexpr int kPlaneA = 444, kPlaneB = 284;
constexpr int kLkSmemFloats = 2 * kPlaneA;
constexpr float kExactBound = 16760000.f;      // < 2^24 by more than the rounding of the float bound itself

// kP = 0: run-time pitch (any working width); kP > 0: the tap offsets are immediates.
template <int kWarpsPerBlock, int kMinBlocks, int kP>
__global__ void __launch_bounds__(kWarpsPerBlock * 32, kMinBlocks)
lk_chain_kernel(const uint8_t* __restrict__ prev_pyr, const uint8_t* __restrict__ next_pyr,
                size_t prev_stride, size_t next_stride, PyrDesc d,
                const float2* __restrict__ pts, const int* __restrict__ counts,
                float2* __restrict__ out_pts, uint8_t* __restrict__ status) {
    __shared__ __align__(16) float smem_all[kWarpsPerBlock][kLkSmemFloats];
    const int frame = blockIdx.y;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int fi = blockIdx.x * kWarpsPerBlock + warp;
    if (fi >= counts[frame]) return;
    float* sm = smem_all[warp];
    const unsigned full = 0xffffffffu;
    const uint8_t* pI = prev_pyr + (size_t)frame * prev_stride;
    const uint8_t* pJ = next_pyr + (size_t)frame * next_stride;
    const float2 pt = pts[(size_t)frame * kMaxCorners + fi];

    // ---- the two strips of this lane (strip = 7 rows of one window column) ------------------------
    const bool isP = lane < 24;
    int q0, c0, q1, c1;
    bool v1 = true;                                            // lane 31: its second strip aliases strip (2, 20) with zero derivatives
    if (isP) {
        const int r = lane & 7;
        q0 = q1 = lane >> 3;
        c0 = (r & 3) + 2 * (r & 4);                            // 0..3, 8..11
        c1 = c0 + 4;
    } else {
        const int i0 = 2 * (lane - 24);
        int i1 = i0 + 1;
        v1 = i1 < 15;
        if (!v1) i1 = 14;
        q0 = i0 / 5; c0 = 16 + i0 % 5;
        q1 = i1 / 5; c1 = 16 + i1 % 5;
    }
    const int chain = isP ? lane & 3 : 4;

    float outx = 0.f, outy = 0.f;
    int st = 1;
    const float half = (float)(kLkWin - 1) * 0.5f;

#pragma unroll 1
    for (int L = d.nlev - 1; L >= 0; --L) {
        const int cols = d.w[L], rows = d.h[L];
        const int P = kP > 0 ? kP : d.pitch[L];
        const size_t org = (size_t)kLkPad * P + kLkPad;          // padded offset of image pixel (0,0)
        const unsigned* I = reinterpret_cast<const unsigned*>(pI + d.qoff[L]) + org;      // bilinear quads of the previous frame
        const unsigned* dI = reinterpret_cast<const unsigned*>(pI + d.doff[L]) + org;    // {dx, dy} short2
        const unsigned* J = reinterpret_cast<const unsigned*>(pJ + d.qoff[L]) + org;      // bilinear quads of the next frame
        const int so0 = kStripLen * q0 * P + c0, so1 = kStripLen * q1 * P + c1;
        const float lscale = (float)(1. / (1 << L));
        float px = __fmul_rn(pt.x, lscale), py = __fmul_rn(pt.y, lscale);
        float nx, ny;
        if (L == d.nlev - 1) { nx = px; ny = py; }
        else { nx = __fmul_rn(outx, 2.f); ny = __fmul_rn(outy, 2.f); }
        outx = nx; outy = ny;
        px = __fsub_rn(px, half); py = __fsub_rn(py, half);
        const int ix = (int)floorf(px), iy = (int)floorf(py);
        if (ix < -kLkWin || ix >= cols || iy < -kLkWin || iy >= rows) {
            if (L == 0) st = 0;
            continue;
        }
        int w00, w01, w10, w11;
        {
            const float a = __fsub_rn(px, (float)ix), b = __fsub_rn(py, (float)iy);
            const float ia = __fsub_rn(1.f, a), ib = __fsub_rn(1.f, b);
            w00 = __float2int_rn(__fmul_rn(__fmul_rn(ia, ib), 16384.f));
            w01 = __float2int_rn(__fmul_rn(__fmul_rn(a, ib), 16384.f));
            w10 = __float2int_rn(__fmul_rn(__fmul_rn(ia, b), 16384.f));
            w11 = 16384 - w00 - w01 - w10;
        }
        const unsigned wt01 = pack_w(w00, w01), wt23 = pack_w(w10, w11);

        // ---- template patch into registers: 2^23 + I (Q5), Ix, Iy as floats (all exact integers) ------
        float Iw[2 * kStripLen], Ix[2 * kStripLen], Iy[2 * kStripLen];
        {
            const int wo = iy * P + ix;
#pragma unroll
            for (int b = 0; b < 2; ++b) {
                const int so = b ? so1 : so0;
                const unsigned* Ip = pin(I + (wo + so));
                const unsigned* Dp = pin(dI + (wo + so));
                if (w00 == (1 << 14)) {
                    // integer window origin (always at level 0: Shi-Tomasi corners are integer-valued): the bilinear taps
                    // collapse to the pixel itself -- (16384 p + 256) >> 9 == 32 p, (16384 d + 8192) >> 14 == d
#pragma unroll
                    for (int t = 0; t < kStripLen; ++t) {
                        const int s = b * kStripLen + t;
                        const unsigned qi = __ldg(Ip + t * P);
                        const unsigned d00 = __ldg(Dp + t * P);
                        Iw[s] = __int_as_float(0x4B000000 + ((int)(qi & 0xffu) << 5));
                        Ix[s] = small_int_to_float((int)(short)(d00 & 0xffffu));
                        Iy[s] = small_int_to_float((int)d00 >> 16);
                    }
                } else {
                    // derivative rows 0..7 of the strip, two columns: the lower taps of row t are the upper taps of row t + 1
                    unsigned dl[kStripLen + 1], dr[kStripLen + 1];
#pragma unroll
                    for (int t = 0; t <= kStripLen; ++t) { dl[t] = __ldg(Dp + t * P); dr[t] = __ldg(Dp + t * P + 1); }
#pragma unroll
                    for (int t = 0; t < kStripLen; ++t) {
                        const int s = b * kStripLen + t;
                        // the 2x2 neighbourhood in one word: 16-bit weights x 8-bit pixels, two dp2a
                        const unsigned qi = __ldg(Ip + t * P);
                        const int iv = dp2a_lo_su(wt01, qi, dp2a_hi_su(wt23, qi, 1 << 8));
                        const unsigned d00 = dl[t], d01 = dr[t], d10 = dl[t + 1], d11 = dr[t + 1];
                        const int xv = (int)(short)(d00 & 0xffffu) * w00 + (int)(short)(d01 & 0xffffu) * w01 +
                                       (int)(short)(d10 & 0xffffu) * w10 + (int)(short)(d11 & 0xffffu) * w11;
                        const int yv = ((int)d00 >> 16) * w00 + ((int)d01 >> 16) * w01 + ((int)d10 >> 16) * w10 + ((int)d11 >> 16) * w11;
                        Iw[s] = __int_as_float(0x4B000000 + (iv >> 9));
                        Ix[s] = small_int_to_float((xv + (1 << 13)) >> 14);
                        Iy[s] = small_int_to_float((yv + (1 << 13)) >> 14);
                    }
                }
            }
            if (!v1) {
#pragma unroll
                for (int t = 0; t < kStripLen; ++t) { Ix[kStripLen + t] = 0.f; Iy[kStripLen + t] = 0.f; }
            }
        }
        // ---- 2x2 normal matrix: OpenCV's five float chains per sum, replayed by lanes 0..14 -----------
        float A11, A12, A22;
        {
            {
                const LaneGeo g = lane_geo(lane);
                float* wx = sm + g.oa;
#pragma unroll
                for (int t = 0; t < kStripLen; ++t) {
                    wx[t * g.sa] = Ix[t];
                    wx[kPlaneA + t * g.sa] = Iy[t];
                }
                if (v1) {
                    float* wy = sm + g.ob;
#pragma unroll
                    for (int t = 0; t < kStripLen; ++t) {
                        wy[t * g.sa] = Ix[kStripLen + t];
                        wy[kPlaneA + t * g.sa] = Iy[kStripLen + t];
                    }
                }
                if (lane < 3) { sm[441 + lane] = 0.f; sm[kPlaneA + 441 + lane] = 0.f; }
            }
            __syncwarp();
            float acc = 0.f;
            if (lane < 15) {
                int rs, rc;
                replay_geo(lane, rs, rc);
                const int cb = rc < 4 ? 84 * rc : 336;
                const float4* a4 = reinterpret_cast<const float4*>(sm + (rs == 2 ? kPlaneA : 0) + cb);
                const float4* b4 = reinterpret_cast<const float4*>(sm + (rs == 0 ? 0 : kPlaneA) + cb);
                // the products are exact (< 2^24), so fma(a, b, acc) == acc + a * b as OpenCV's mul + add computes it
#define VSTAB_LK_A_STEP(i) { const float4 a = a4[i], b = b4[i]; acc = __fmaf_rn(a.x, b.x, acc); acc = __fmaf_rn(a.y, b.y, acc); \
                             acc = __fmaf_rn(a.z, b.z, acc); acc = __fmaf_rn(a.w, b.w, acc); }
#pragma unroll 3
                for (int i = 0; i < 21; ++i) VSTAB_LK_A_STEP(i)          // 84 terms: all chains
                if (rc == 4) {
#pragma unroll 3
                    for (int i = 21; i < 27; ++i) VSTAB_LK_A_STEP(i)     // the scalar chain has 105 (+ 3 zero pads)
                }
#undef VSTAB_LK_A_STEP
            }
            __syncwarp();
            float s[3];
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const float e0 = __shfl_sync(full, acc, 5 * k), e1 = __shfl_sync(full, acc, 5 * k + 1), e2 = __shfl_sync(full, acc, 5 * k + 2),
                            e3 = __shfl_sync(full, acc, 5 * k + 3), e4 = __shfl_sync(full, acc, 5 * k + 4);
                s[k] = __fmul_rn(combine_chains(e0, e1, e2, e3, e4), 1.f / (float)(1 << 20));
            }
            A11 = s[0]; A12 = s[1]; A22 = s[2];
        }
        float D = __fsub_rn(__fmul_rn(A11, A22), __fmul_rn(A12, A12));
        {
            const float dd = __fsub_rn(A11, A22);
            const float rad = __fsqrt_rn(__fadd_rn(__fmul_rn(dd, dd), __fmul_rn(__fmul_rn(4.f, A12), A12)));
            const float min_eig = __fdiv_rn(__fsub_rn(__fadd_rn(A22, A11), rad), (float)(2 * kPix));
            if ((double)min_eig < 1e-4 || D < 1.1920928955078125e-7f) {   // minEigThreshold is a double
                if (L == 0) st = 0;
                continue;
            }
        }
        D = __fdiv_rn(1.f, D);
        nx = __fsub_rn(nx, half); ny = __fsub_rn(ny, half);
        float pdx = 0.f, pdy = 0.f;
#pragma unroll 1
        for (int j = 0; j < kLkMaxIter; ++j) {
            const int jx = (int)floorf(nx), jy = (int)floorf(ny);
            if (jx < -kLkWin || jx >= cols || jy < -kLkWin || jy >= rows) {
                if (L == 0) st = 0;
                break;
            }
            unsigned vt01, vt23;
            {
                const float a = __fsub_rn(nx, (float)jx), b = __fsub_rn(ny, (float)jy);
                const float ia = __fsub_rn(1.f, a), ib = __fsub_rn(1.f, b);
                const int v00 = __float2int_rn(__fmul_rn(__fmul_rn(ia, ib), 16384.f));
                const int v01 = __float2int_rn(__fmul_rn(__fmul_rn(a, ib), 16384.f));
                const int v10 = __float2int_rn(__fmul_rn(__fmul_rn(ia, b), 16384.f));
                const int v11 = 16384 - v00 - v01 - v10;
                vt01 = pack_w(v00, v01); vt23 = pack_w(v10, v11);
            }
            const int jo = jy * P + jx;
            const unsigned* Jp0 = pin(J + (jo + so0));
            const unsigned* Jp1 = pin(J + (jo + so1));
            unsigned q[2 * kStripLen];
#pragma unroll
            for (int t = 0; t < kStripLen; ++t) { q[t] = __ldg(Jp0 + t * P); q[kStripLen + t] = __ldg(Jp1 + t * P); }
            // mismatch I_t = J - I (exact, |.| <= 8160) and the lane's share of b1 = sum I_t Ix, b2 = sum I_t Iy in float: exact
            // while the bound (sum of |terms|, same instruction with the free |.| modifiers) stays below 2^24
            float acc1 = 0.f, acc2 = 0.f, bn1 = 0.f, bn2 = 0.f;
#pragma unroll
            for (int s = 0; s < 2 * kStripLen; ++s) {
                const int jv = dp2a_lo_su(vt01, q[s], dp2a_hi_su(vt23, q[s], 1 << 8)) >> 9;
                const float fd = __fsub_rn(__int_as_float(0x4B000000 + jv), Iw[s]);
                acc1 = __fmaf_rn(fd, Ix[s], acc1);
                acc2 = __fmaf_rn(fd, Iy[s], acc2);
                bn1 = __fmaf_rn(fabsf(fd), fabsf(Ix[s]), bn1);
                bn2 = __fmaf_rn(fabsf(fd), fabsf(Iy[s]), bn2);
            }
            float b1, b2;
            {
                // Every partial sum of a set of terms lies in [-P-, P+] (P+ / P- = sum of its positive / |negative| terms), and the
                // lane has both for free: P+ = (bound + sum) / 2, P- = (bound - sum) / 2.  Quantised upwards, the larger of b1's and
                // b2's, packed as two 16-bit fields so that one redux.sync adds both over the warp or over a chain.
                const bool lane_exact = fmaxf(bn1, bn2) < kExactBound;            // else the lane's own float sums may have rounded
                const float pp = fmaxf(__fadd_rn(bn1, acc1), __fadd_rn(bn2, acc2));   // 2 P+
                const float pm = fmaxf(__fsub_rn(bn1, acc1), __fsub_rn(bn2, acc2));   // 2 P-
                // warp-wide fields in units of 2^15 (<= 513 per lane), chain fields in units of 2^13 (<= 2049 per lane, <= 8 lanes)
                const int wp = lane_exact ? __float2int_rz(__fmul_rn(pp, 1.f / 65536.f)) + 1 : 600;
                const int wm = lane_exact ? __float2int_rz(__fmul_rn(pm, 1.f / 65536.f)) + 1 : 600;
                const unsigned tot = __reduce_add_sync(full, (unsigned)wp | ((unsigned)wm << 16));
                if ((tot & 0xffffu) <= 511u && (tot >> 16) <= 511u) {
                    // tier 0: no partial sum of any order reaches 2^24 (511 * 2^15 < 2^24)
                    b1 = (float)__reduce_add_sync(full, __float2int_rn(acc1));
                    b2 = (float)__reduce_add_sync(full, __float2int_rn(acc2));
                } else {
                    const int cp = lane_exact ? __float2int_rz(__fmul_rn(pp, 1.f / 16384.f)) + 1 : 2100;
                    const int cm = lane_exact ? __float2int_rz(__fmul_rn(pm, 1.f / 16384.f)) + 1 : 2100;
                    const unsigned cpk = (unsigned)cp | ((unsigned)cm << 16);
                    bool ok = true;
#pragma unroll
                    for (int c = 0; c < 5; ++c) {
                        const unsigned r = __reduce_add_sync(full, chain == c ? cpk : 0u);
                        ok = ok && (r & 0xffffu) <= 2047u && (r >> 16) <= 2047u;      // 2047 * 2^13 < 2^24
                    }
                    float e1[5], e2[5];
                    if (ok) {
                        // tier 1: every chain is exact; OpenCV's four float additions on top
                        const int a1 = __float2int_rn(acc1), a2 = __float2int_rn(acc2);
#pragma unroll
                        for (int c = 0; c < 5; ++c) {
                            e1[c] = (float)__reduce_add_sync(full, chain == c ? a1 : 0);
                            e2[c] = (float)__reduce_add_sync(full, chain == c ? a2 : 0);
                        }
                    } else {
                        // tier 2: terms in chain order through shared memory (the integer pair sums of OpenCV's v_dotprod for the
                        // SIMD chains), then lanes 0..9 replay the sequential float additions.  The taps are read again (L1).
                        int rs, rc;
                        replay_geo(lane, rs, rc);
                        float* rdB = sm + (rs & 1) * kPlaneB + (rc < 4 ? 44 * rc : 176);
                        if (lane < 10) {
                            if (rc < 4) { rdB[42] = 0.f; rdB[43] = 0.f; }
                            else { rdB[105] = 0.f; rdB[106] = 0.f; rdB[107] = 0.f; }
                        }
                        {
                            const LaneGeo g = lane_geo(lane);
                            float* w0 = sm + g.ta;
                            float* w1 = sm + g.tb;
#pragma unroll
                            for (int t = 0; t < kStripLen; ++t) {
                                const unsigned qa = __ldg(Jp0 + t * P), qb = __ldg(Jp1 + t * P);
                                const int d0 = (dp2a_lo_su(vt01, qa, dp2a_hi_su(vt23, qa, 1 << 8)) >> 9) - (__float_as_int(Iw[t]) - 0x4B000000);
                                const int d1 = (dp2a_lo_su(vt01, qb, dp2a_hi_su(vt23, qb, 1 << 8)) >> 9) - (__float_as_int(Iw[kStripLen + t]) - 0x4B000000);
                                const int u1 = d0 * __float2int_rn(Ix[t]), u2 = d0 * __float2int_rn(Iy[t]);
                                const int g1 = d1 * __float2int_rn(Ix[kStripLen + t]), g2 = d1 * __float2int_rn(Iy[kStripLen + t]);
                                w0[t * g.sb] = (float)(isP ? u1 + g1 : u1);
                                w0[kPlaneB + t * g.sb] = (float)(isP ? u2 + g2 : u2);
                                if (!isP && v1) {
                                    w1[t * g.sb] = (float)g1;
                                    w1[kPlaneB + t * g.sb] = (float)g2;
                                }
                            }
                        }
                        __syncwarp();
                        float acc = 0.f;
                        if (lane < 10) {
                            const float4* p4 = reinterpret_cast<const float4*>(rdB);
#define VSTAB_LK_B_STEP(i) { const float4 v = p4[i]; acc = __fadd_rn(acc, v.x); acc = __fadd_rn(acc, v.y); acc = __fadd_rn(acc, v.z); acc = __fadd_rn(acc, v.w); }
#pragma unroll 4
                            for (int i = 0; i < 11; ++i) VSTAB_LK_B_STEP(i)          // 42 pair terms (+ 2 zero pads): all chains
                            if (rc == 4) {
#pragma unroll 4
                                for (int i = 11; i < 27; ++i) VSTAB_LK_B_STEP(i)     // the scalar chain has 105 (+ 3 zero pads)
                            }
#undef VSTAB_LK_B_STEP
                        }
                        __syncwarp();
#pragma unroll
                        for (int c = 0; c < 5; ++c) { e1[c] = __shfl_sync(full, acc, c); e2[c] = __shfl_sync(full, acc, 5 + c); }
                    }
                    b1 = combine_chains(e1[0], e1[1], e1[2], e1[3], e1[4]);
                    b2 = combine_chains(e2[0], e2[1], e2[2], e2[3], e2[4]);
                }
            }
            b1 = __fmul_rn(b1, 1.f / (float)(1 << 20));
            b2 = __fmul_rn(b2, 1.f / (float)(1 << 20));
            const float ddx = __fmul_rn(__fsub_rn(__fmul_rn(A12, b2), __fmul_rn(A22, b1)), D);
            const float ddy = __fmul_rn(__fsub_rn(__fmul_rn(A12, b1), __fmul_rn(A11, b2)), D);
            nx = __fadd_rn(nx, ddx); ny = __fadd_rn(ny, ddy);
            outx = __fadd_rn(nx, half); outy = __fadd_rn(ny, half);
            // delta.ddot(delta) <= criteria.epsilon^2 with Point2f::ddot in double: decided in float when the float value
            // is outside a 1e-5 relative band around the threshold (float error <= 2^-22), in double inside it
            {
                const float sf = __fmaf_rn(ddx, ddx, __fmul_rn(ddy, ddy));
                bool conv = sf < 0.99999e-4f;
                if (!conv && sf < 1.00001e-4f) conv = (double)ddx * (double)ddx + (double)ddy * (double)ddy <= 0.01 * 0.01;
                if (conv) break;
            }
            // float < 0.01 (a double): 0x3C23D70A = 0.0099999998 is the largest float below it
            if (j > 0 && fabsf(__fadd_rn(ddx, pdx)) <= 0.01f && fabsf(__fadd_rn(ddy, pdy)) <= 0.01f) {
                outx = __fsub_rn(outx, __fmul_rn(ddx, 0.5f));
                outy = __fsub_rn(outy, __fmul_rn(ddy, 0.5f));
                break;
            }
            pdx = ddx; pdy = ddy;
        }
        // the `err` block of OpenCV's LKTrackerInvoker (the reference passes an err vector,
        // stabilizer.cpp:192-195): at level 0 a still-valid point whose final window origin lies
        // outside the image loses its status (coordinates are kept).
        if (L == 0 && st) {
            const int fx = (int)floorf(__fsub_rn(outx, half)), fy = (int)floorf(__fsub_rn(outy, half));
            if (fx < -kLkWin || fx >= cols || fy < -kLkWin || fy >= rows) st = 0;
        }
    }
    if (lane == 0) {
        out_pts[(size_t)frame * kMaxCorners + fi] = make_float2(outx, outy);
        status[(size_t)frame * kMaxCorners + fi] = (uint8_t)st;
    }
}

template <int kWarpsPerBlock, int kMinBlocks>
void launch_chain(int P, int nframes, cudaStream_t st, const uint8_t* prev_pyr, const uint8_t* next_pyr, size_t prev_stride,
                  size_t next_stride, const PyrDesc& d, const float2* pts, const int* counts, float2* out_pts, uint8_t* status) {
    const int T = kWarpsPerBlock * 32;
    const dim3 grid((kMaxCorners + kWarpsPerBlock - 1) / kWarpsPerBlock, nframes);
    // working widths 640 (wh 360 of 16:9 input), 1920, 3840 (+ 2 * kLkPad) get immediate tap offsets
    if (P == 688) lk_chain_kernel<kWarpsPerBlock, kMinBlocks, 688><<<grid, T, 0, st>>>(prev_pyr, next_pyr, prev_stride, next_stride, d, pts, counts, out_pts, status);
    else if (P == 1968) lk_chain_kernel<kWarpsPerBlock, kMinBlocks, 1968><<<grid, T, 0, st>>>(prev_pyr, next_pyr, prev_stride, next_stride, d, pts, counts, out_pts, status);
    else if (P == 3888) lk_chain_kernel<kWarpsPerBlock, kMinBlocks, 3888><<<grid, T, 0, st>>>(prev_pyr, next_pyr, prev_stride, next_stride, d, pts, counts, out_pts, status);
    else lk_chain_kernel<kWarpsPerBlock, kMinBlocks, 0><<<grid, T, 0, st>>>(prev_pyr, next_pyr, prev_stride, next_stride, d, pts, counts, out_pts, status);
}

}  // namespace

void launch_lk(const uint8_t* prev_pyr, const uint8_t* next_pyr, size_t prev_stride, size_t next_stride,
               const PyrDesc& d, const float2* pts, const int* counts, int nframes,
               float2* out_pts, uint8_t* status, cudaStream_t st) {
    if (nframes <= 0) return;
    count_launch(1);
    // One warp per CTA: a CTA's registers and shared memory are held until its slowest feature converges, so one-warp
    // CTAs refill soonest (round 1: 4 / 2 / 1 warps per CTA 1.73 / 1.71 / 1.66 ms per 256 frames).
    bool uniform = true;
    for (int l = 1; l < d.nlev; ++l) uniform = uniform && d.pitch[l] == d.pitch[0];
    const int P = uniform ? d.pitch[0] : 0;
    // 16 CTAs per SM: 128 registers per thread (min blocks per SM = 65536 / (registers * threads per CTA))
    launch_chain<1, 16>(P, nframes, st, prev_pyr, next_pyr, prev_stride, next_stride, d, pts, counts, out_pts, status);
}

}  // namespace vstabk
