// K11: SIFT keypoints + 128-D descriptors
//   cv::SIFT::create(2500, 3, 0.04, 5, 1.2)->detectAndCompute      /root/reference/src/stabilizer.cpp:496-506,
//   :549-553, :572-574, :614-615;  filterKeypointByRelativeSize(0.05)  :290-309, :617-621
// Follows OpenCV's float pipeline (SURVEY A.12): 2x linear upsample + blur to sigma 1.2, per octave six
// Gaussians (incremental sigmas, kernel size cvRound(8 sigma + 1) | 1, BORDER_REFLECT_101), next octave
// = nearest decimation of Gaussian #3, DoG 3x3x3 extrema above floor(0.5*0.04/3*255), <= 5 quadratic
// refinement steps, contrast and edge tests, 36-bin orientation histogram with extra keypoints for
// peaks >= 0.8 max, removal of duplicates, retainBest(2500) by response with ties kept, 4x4x8
// trilinear descriptor, normalise -> clip 0.2 -> normalise -> x512 -> saturate to u8.
// Floating point, not bit-pinned: parity is stated at the homography level (<= 0.1 px) and by keypoint
// overlap, as in SURVEY 7.2(3).  The DoG pyramid is never materialised (differences of the Gaussian
// levels are recomputed where needed: the same float values).
#include <cub/device/device_radix_sort.cuh>
#include <cmath>
#include <vector>
#include "kernels.h"

namespace vstabk {
namespace {

constexpr int kLayers = 3;                // nOctaveLayers
constexpr int kGauss = kLayers + 3;       // Gaussians per octave
constexpr int kBorder = 5;                // SIFT_IMG_BORDER
constexpr int kMaxRadius = 12;            // largest Gaussian half-width used (sigma 2.32 -> 21 taps -> 10)
constexpr float kContrastThr = 0.04f, kEdgeThr = 5.f, kSigma = 1.2f;

struct SiftOctaves {
    int n;
    int w[kSiftMaxOctaves], h[kSiftMaxOctaves];
    size_t off[kSiftMaxOctaves];          // float offset of Gaussian 0 of octave o; Gaussian i at off + i*w*h
};

__constant__ float c_gk[kGauss + 1][2 * kMaxRadius + 1];   // [0] = initial blur, [1..5] = incremental blurs
__constant__ int c_gr[kGauss + 1];

// ---------------------------------------------------------------- base image: u8 -> float, 2x INTER_LINEAR
// cv::resize(INTER_LINEAR) by exactly 2: output 2i takes source columns (i-1, i) with weights (.25, .75), output 2i+1 takes
// (i, i+1) with (.75, .25), clamped at the borders; the same along y.  All products and sums of u8 values with these weights
// are exact in fp32, so the order of evaluation does not matter.  One thread per SOURCE pixel: 9 bytes in, a 2 x 2 block out.
__global__ void __launch_bounds__(256)
sift_upsample_kernel(const uint8_t* __restrict__ gray, int w, int h, float* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y;
    if (i >= w) return;
    const int il = max(i - 1, 0), ir = min(i + 1, w - 1);
    const int jr[3] = {max(j - 1, 0), j, min(j + 1, h - 1)};
    float hl[3], hr[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        const uint8_t* row = gray + (size_t)jr[r] * w;
        const float a = (float)__ldg(row + il), b = (float)__ldg(row + i), c = (float)__ldg(row + ir);
        hl[r] = a * 0.25f + b * 0.75f;
        hr[r] = b * 0.75f + c * 0.25f;
    }
    const int W = 2 * w;
    float2* o0 = reinterpret_cast<float2*>(out + (size_t)(2 * j) * W + 2 * i);
    float2* o1 = reinterpret_cast<float2*>(out + (size_t)(2 * j + 1) * W + 2 * i);
    *o0 = make_float2(hl[0] * 0.25f + hl[1] * 0.75f, hr[0] * 0.25f + hr[1] * 0.75f);
    *o1 = make_float2(hl[1] * 0.75f + hl[2] * 0.25f, hr[1] * 0.75f + hr[2] * 0.25f);
}

// ---------------------------------------------------------------- separable Gaussian blur (float), REFLECT_101
constexpr int GBX = 64, GBY = 16;
__global__ void __launch_bounds__(256)
sift_blur_kernel(const float* __restrict__ src, float* __restrict__ dst, int w, int h, int ki) {
    extern __shared__ float sm[];
    const int R = c_gr[ki];
    const int tw = GBX + 2 * R, th = GBY + 2 * R;
    float* tile = sm;                       // th x tw
    float* rowf = sm + th * tw;             // th x GBX
    const int x0 = blockIdx.x * GBX, y0 = blockIdx.y * GBY;
    for (int i = threadIdx.x; i < th * tw; i += 256) {
        const int r = i / tw, c = i - r * tw;
        const int yy = reflect101_multi(y0 + r - R, h), xx = reflect101_multi(x0 + c - R, w);
        tile[i] = src[(size_t)yy * w + xx];
    }
    __syncthreads();
    const float* k = c_gk[ki];
    for (int i = threadIdx.x; i < th * GBX; i += 256) {
        const int r = i / GBX, c = i - r * GBX;
        const float* t = tile + r * tw + c;
        float s = 0.f;
        for (int j = 0; j <= 2 * R; ++j) s += t[j] * k[j];
        rowf[i] = s;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < GBY * GBX; i += 256) {
        const int r = i / GBX, c = i - r * GBX;
        const int x = x0 + c, y = y0 + r;
        if (x >= w || y >= h) continue;
        float s = 0.f;
        for (int j = 0; j <= 2 * R; ++j) s += rowf[(r + j) * GBX + c] * k[j];
        dst[(size_t)y * w + x] = s;
    }
}

// Same blur for a radius known at compile time (the six radii SIFT's sigmas produce): 64 x 64 output tile, reflect
// indices from small tables, the horizontal pass register-blocked 4 outputs wide on 16-byte shared-memory loads, the
// vertical pass as a register window sliding down 16 rows of a column; taps are accumulated in the same order as the
// generic kernel (bit-identical results).
constexpr int TBX = 64, TBY = 64;
template <int R>
__global__ void __launch_bounds__(256)
sift_blur_t_kernel(const float* __restrict__ src, float* __restrict__ dst, int w, int h, int ki) {
    constexpr int TW = TBX + 2 * R, TH = TBY + 2 * R, TWS = (TW + 3) & ~3, NT = 2 * R + 1;
    extern __shared__ __align__(16) float sm[];
    float* tile = sm;                       // TH x TWS
    float* rowf = sm + TH * TWS;            // TH x TBX
    __shared__ int sx[TW], sy[TH];
    const int x0 = blockIdx.x * TBX, y0 = blockIdx.y * TBY;
    const int tid = threadIdx.x;
    for (int i = tid; i < TW; i += 256) sx[i] = reflect101_multi(x0 + i - R, w);
    for (int i = tid; i < TH; i += 256) sy[i] = reflect101_multi(y0 + i - R, h) * w;      // (< 2^31: at most 7680 x 4320)
    __syncthreads();
    {
        // all loads of a thread in flight together (one memory round trip per tile instead of one per element)
        constexpr int NE = (TH * TW + 255) / 256;
        float v[NE];
#pragma unroll
        for (int e = 0; e < NE; ++e) {
            const int i = tid + e * 256;
            const int r = i / TW, c = i - r * TW;
            v[e] = i < TH * TW ? __ldg(src + sy[r] + sx[c]) : 0.f;
        }
#pragma unroll
        for (int e = 0; e < NE; ++e) {
            const int i = tid + e * 256;
            const int r = i / TW, c = i - r * TW;
            if (i < TH * TW) tile[r * TWS + c] = v[e];
        }
    }
    __syncthreads();
    float k[NT];
#pragma unroll
    for (int j = 0; j < NT; ++j) k[j] = c_gk[ki][j];
    // horizontal: TH rows x 16 groups of 4 outputs
    for (int it = tid; it < TH * (TBX / 4); it += 256) {
        const int r = it / (TBX / 4), c4 = (it - r * (TBX / 4)) * 4;
        constexpr int NV = (NT + 3 + 3) / 4;                    // float4 loads covering taps c4 .. c4 + NT + 2
        float v[NV * 4];
        const float4* t4 = reinterpret_cast<const float4*>(tile + r * TWS + c4);
#pragma unroll
        for (int q = 0; q < NV; ++q) {
            const float4 f = t4[q];
            v[4 * q] = f.x; v[4 * q + 1] = f.y; v[4 * q + 2] = f.z; v[4 * q + 3] = f.w;
        }
        float o[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            float s = 0.f;
#pragma unroll
            for (int j = 0; j < NT; ++j) s += v[u + j] * k[j];
            o[u] = s;
        }
        *reinterpret_cast<float4*>(rowf + r * TBX + c4) = make_float4(o[0], o[1], o[2], o[3]);
    }
    __syncthreads();
    // vertical: column c, 16 consecutive output rows per thread
    {
        const int c = tid & (TBX - 1), r0 = (tid / TBX) * 16;
        float v[16 + 2 * R];
#pragma unroll
        for (int i = 0; i < 16 + 2 * R; ++i) v[i] = rowf[(r0 + i) * TBX + c];
        const int x = x0 + c;
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            float s = 0.f;
#pragma unroll
            for (int j = 0; j < NT; ++j) s += v[i + j] * k[j];
            const int y = y0 + r0 + i;
            if (x < w && y < h) dst[(size_t)y * w + x] = s;
        }
    }
}

template <int R>
static void launch_blur_t(const float* src, float* dst, int w, int h, int ki, cudaStream_t st) {
    constexpr int TW = TBX + 2 * R, TH = TBY + 2 * R, TWS = (TW + 3) & ~3;
    constexpr int smem = (int)(sizeof(float) * (TH * TWS + TH * TBX));
    static PerDeviceOnce once;
    once.run([] { cudaFuncSetAttribute(sift_blur_t_kernel<R>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem); });
    sift_blur_t_kernel<R><<<dim3((w + TBX - 1) / TBX, (h + TBY - 1) / TBY), 256, smem, st>>>(src, dst, w, h, ki);
}

__global__ void __launch_bounds__(256)
sift_decimate_kernel(const float* __restrict__ src, int sw, float* __restrict__ dst, int dw, int dh) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= dw || y >= dh) return;
    dst[(size_t)y * dw + x] = src[(size_t)(2 * y) * sw + 2 * x];
}

// ---------------------------------------------------------------- DoG extrema
// candidate = octave << 56 | layer << 48 | r << 24 | c
__global__ void __launch_bounds__(256)
sift_extrema_kernel(const float* __restrict__ pyr, SiftOctaves O, int o, int threshold,
                    unsigned long long* __restrict__ cand, int* __restrict__ ncand, int cap) {
    const int w = O.w[o], h = O.h[o];
    const int layer = 1 + blockIdx.z;                      // DoG layer 1..3
    const size_t plane = (size_t)w * h;
    const float* g = pyr + O.off[o] + (size_t)(layer - 1) * plane;   // Gaussians layer-1 .. layer+2
    const int x = kBorder + blockIdx.x * blockDim.x + threadIdx.x;
    const int y = kBorder + blockIdx.y;
    bool is_ext = false;
    if (x < w - kBorder && y < h - kBorder) {
        const size_t p = (size_t)y * w + x;
        const float val = g[2 * plane + p] - g[plane + p];
        if (fabsf(val) > (float)threshold) {
            bool mx = val > 0.f, mn = val < 0.f;
#pragma unroll
            for (int dl = 0; dl < 3 && (mx || mn); ++dl) {
                const float* a = g + (size_t)dl * plane;
                const float* b = a + plane;
#pragma unroll
                for (int dy = -1; dy <= 1; ++dy)
#pragma unroll
                    for (int dx = -1; dx <= 1; ++dx) {
                        const size_t q = p + (long)dy * w + dx;
                        const float v = b[q] - a[q];
                        mx = mx && val >= v;
                        mn = mn && val <= v;
                    }
            }
            is_ext = mx || mn;
        }
    }
    const unsigned ball = __ballot_sync(0xffffffffu, is_ext);
    if (ball) {
        const int lane = threadIdx.x & 31;
        int pos0 = 0;
        if (lane == 0) pos0 = atomicAdd(ncand, __popc(ball));
        pos0 = __shfl_sync(0xffffffffu, pos0, 0);
        if (is_ext) {
            const int pos = pos0 + __popc(ball & ((1u << lane) - 1u));
            if (pos < cap)
                cand[pos] = ((unsigned long long)o << 56) | ((unsigned long long)layer << 48) | ((unsigned long long)y << 24) |
                            (unsigned long long)x;
        }
    }
}

// Same test on shared-memory tiles: one CTA stages the 5 DoG layers of a 64 x 16 tile (+1 halo) -- every Gaussian
// sample is read once per tile instead of up to 27 times per layer -- and every thread tests 4 rows x 3 layers.
constexpr int EXW = 64, EXH = 16;
__global__ void __launch_bounds__(256)
sift_extrema_tile_kernel(const float* __restrict__ pyr, SiftOctaves O, int o, int threshold,
                         unsigned long long* __restrict__ cand, int* __restrict__ ncand, int cap) {
    // tile rows start at x0 - 1 = kBorder - 1 + 64 bx, a multiple of 4 floats: staged as float4 (17 per row, row stride 68)
    constexpr int TH = EXH + 2, TWV = (EXW + 2 + 3) / 4, TWP = 4 * TWV, NE = (TWV * TH + 255) / 256;
    static_assert((kBorder - 1) % 4 == 0, "tile rows must start on a 16-byte boundary");
    __shared__ __align__(16) float D[kGauss - 1][TH][TWP];
    const int w = O.w[o], h = O.h[o];
    const size_t plane = (size_t)w * h;
    const float* g = pyr + O.off[o];
    const int x0 = kBorder + blockIdx.x * EXW, y0 = kBorder + blockIdx.y * EXH;
    const int tid = threadIdx.x;
    {
        const bool vec_ok = (w & 3) == 0;
        float4 prev[NE];
#pragma unroll
        for (int l = 0; l < kGauss; ++l) {
            float4 cur[NE];
#pragma unroll
            for (int e = 0; e < NE; ++e) {
                const int i = tid + e * 256;
                const int r = i / TWV, c4 = i - r * TWV;
                cur[e] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (i < TWV * TH) {
                    const int yy = min(y0 - 1 + r, h - 1), xb = x0 - 1 + 4 * c4;
                    const float* rowp = g + (size_t)l * plane + (size_t)yy * w;
                    if (vec_ok && xb + 3 <= w - 1) {
                        cur[e] = __ldg(reinterpret_cast<const float4*>(rowp + xb));
                    } else {
                        cur[e].x = __ldg(rowp + min(xb, w - 1)); cur[e].y = __ldg(rowp + min(xb + 1, w - 1));
                        cur[e].z = __ldg(rowp + min(xb + 2, w - 1)); cur[e].w = __ldg(rowp + min(xb + 3, w - 1));
                    }
                }
            }
            if (l > 0) {
#pragma unroll
                for (int e = 0; e < NE; ++e) {
                    const int i = tid + e * 256;
                    const int r = i / TWV, c4 = i - r * TWV;
                    if (i < TWV * TH)
                        *reinterpret_cast<float4*>(&D[l - 1][r][4 * c4]) =
                            make_float4(cur[e].x - prev[e].x, cur[e].y - prev[e].y, cur[e].z - prev[e].z, cur[e].w - prev[e].w);
                }
            }
#pragma unroll
            for (int e = 0; e < NE; ++e) prev[e] = cur[e];
        }
    }
    __syncthreads();
    const int c = 1 + (tid & (EXW - 1));
    const int x = x0 + c - 1;
    const int lane = tid & 31;
#pragma unroll 1
    for (int rr = 0; rr < 4; ++rr) {
        const int r = 1 + (tid / EXW) * 4 + rr;
        const int y = y0 + r - 1;
#pragma unroll 1
        for (int layer = 1; layer <= kLayers; ++layer) {
            bool is_ext = false;
            if (x < w - kBorder && y < h - kBorder) {
                const float val = D[layer][r][c];
                if (fabsf(val) > (float)threshold) {
                    // own layer first: few samples are 2-D extrema, the two neighbouring layers are only read for those
                    bool mx = val > 0.f, mn = val < 0.f;
#pragma unroll
                    for (int dy = -1; dy <= 1; ++dy)
#pragma unroll
                        for (int dx = -1; dx <= 1; ++dx) {
                            const float v = D[layer][r + dy][c + dx];
                            mx = mx && val >= v;
                            mn = mn && val <= v;
                        }
                    if (mx || mn) {
#pragma unroll
                        for (int dl = -1; dl <= 1; dl += 2)
#pragma unroll
                            for (int dy = -1; dy <= 1; ++dy)
#pragma unroll
                                for (int dx = -1; dx <= 1; ++dx) {
                                    const float v = D[layer + dl][r + dy][c + dx];
                                    mx = mx && val >= v;
                                    mn = mn && val <= v;
                                }
                    }
                    is_ext = mx || mn;
                }
            }
            const unsigned ball = __ballot_sync(0xffffffffu, is_ext);
            if (ball) {
                int pos0 = 0;
                if (lane == 0) pos0 = atomicAdd(ncand, __popc(ball));
                pos0 = __shfl_sync(0xffffffffu, pos0, 0);
                if (is_ext) {
                    const int pos = pos0 + __popc(ball & ((1u << lane) - 1u));
                    if (pos < cap)
                        cand[pos] = ((unsigned long long)o << 56) | ((unsigned long long)layer << 48) | ((unsigned long long)y << 24) |
                                    (unsigned long long)x;
                }
            }
        }
    }
}

// DoG value: layer l (0..4) of octave image set `g0` (Gaussian 0), at (r, c)
VSTAB_D float dogv(const float* __restrict__ g0, size_t plane, int w, int l, int r, int c) {
    const size_t p = (size_t)r * w + c;
    return g0[(size_t)(l + 1) * plane + p] - g0[(size_t)l * plane + p];
}

// 3x3 solve with partial pivoting (Matx33f::solve(DECOMP_LU))
VSTAB_D bool solve3(float A[3][3], float b[3], float x[3]) {
    for (int i = 0; i < 3; ++i) {
        int k = i;
        for (int j = i + 1; j < 3; ++j) if (fabsf(A[j][i]) > fabsf(A[k][i])) k = j;
        if (fabsf(A[k][i]) < 1.1920929e-7f) return false;
        if (k != i) { for (int j = i; j < 3; ++j) { const float t = A[i][j]; A[i][j] = A[k][j]; A[k][j] = t; } const float t = b[i]; b[i] = b[k]; b[k] = t; }
        const float d = -1.f / A[i][i];
        for (int j = i + 1; j < 3; ++j) {
            const float alpha = A[j][i] * d;
            for (int c = i + 1; c < 3; ++c) A[j][c] += alpha * A[i][c];
            b[j] += alpha * b[i];
        }
    }
    for (int i = 2; i >= 0; --i) {
        float s = b[i];
        for (int c = i + 1; c < 3; ++c) s -= A[i][c] * x[c];
        x[i] = s / A[i][i];
    }
    return true;
}

// cv::fastAtan2 (degrees), see orb.cu
VSTAB_D float atan2_deg(float y, float x) {
    const float scale = (float)(180.0 / 3.14159265358979323846);
    const float p1 = 0.9997878412794807f * scale, p3 = -0.3258083974640975f * scale;
    const float p5 = 0.1555786518463281f * scale, p7 = -0.04432655554792128f * scale;
    const float eps = (float)2.2204460492503131e-16;
    const float ax = fabsf(x), ay = fabsf(y);
    float a, c, c2;
    if (ax >= ay) { c = ay / (ax + eps); c2 = c * c; a = (((p7 * c2 + p5) * c2 + p3) * c2 + p1) * c; }
    else { c = ax / (ay + eps); c2 = c * c; a = 90.f - (((p7 * c2 + p5) * c2 + p3) * c2 + p1) * c; }
    if (x < 0) a = 180.f - a;
    if (y < 0) a = 360.f - a;
    return a;
}

struct SiftKp { float x, y, size, angle, response; int octave; };   // == OrbKeypoint layout

// ---------------------------------------------------------------- refine + orientation, one warp per candidate
__global__ void __launch_bounds__(128)
sift_refine_kernel(const float* __restrict__ pyr, SiftOctaves O, const unsigned long long* __restrict__ cand,
                   const int* __restrict__ ncand, int cap, SiftKp* __restrict__ kps, int* __restrict__ nkp, int kcap) {
    __shared__ float hist_s[4][40];
    const int n = min(*ncand, cap);
    const int lane = threadIdx.x & 31, wl = threadIdx.x >> 5;
    // a fixed grid walks the candidate list (the capacity is ~2 M entries at 4K, the list a few tens of thousands)
    for (int ci = blockIdx.x * 4 + wl; ci < n; ci += gridDim.x * 4) {
    __syncwarp();
    const unsigned long long key = cand[ci];
    const int o = (int)(key >> 56);
    int layer = (int)((key >> 48) & 0xff), r = (int)((key >> 24) & 0xffffff), c = (int)(key & 0xffffff);
    const int w = O.w[o], h = O.h[o];
    const size_t plane = (size_t)w * h;
    const float* g0 = pyr + O.off[o];

    // ---- adjustLocalExtrema (lane 0; the rest of the warp waits) --------------------------------
    int ok = 0;
    float xi = 0.f, xr = 0.f, xc = 0.f, contr = 0.f;
    if (lane == 0) {
        const float img_scale = 1.f / 255.f, deriv_scale = img_scale * 0.5f, second_scale = img_scale, cross_scale = img_scale * 0.25f;
        int i = 0;
        bool alive = true;
        for (; i < 5; ++i) {
            const float v2 = dogv(g0, plane, w, layer, r, c) * 2.f;
            float dD[3] = {(dogv(g0, plane, w, layer, r, c + 1) - dogv(g0, plane, w, layer, r, c - 1)) * deriv_scale,
                           (dogv(g0, plane, w, layer, r + 1, c) - dogv(g0, plane, w, layer, r - 1, c)) * deriv_scale,
                           (dogv(g0, plane, w, layer + 1, r, c) - dogv(g0, plane, w, layer - 1, r, c)) * deriv_scale};
            const float dxx = (dogv(g0, plane, w, layer, r, c + 1) + dogv(g0, plane, w, layer, r, c - 1) - v2) * second_scale;
            const float dyy = (dogv(g0, plane, w, layer, r + 1, c) + dogv(g0, plane, w, layer, r - 1, c) - v2) * second_scale;
            const float dss = (dogv(g0, plane, w, layer + 1, r, c) + dogv(g0, plane, w, layer - 1, r, c) - v2) * second_scale;
            const float dxy = (dogv(g0, plane, w, layer, r + 1, c + 1) - dogv(g0, plane, w, layer, r + 1, c - 1) -
                               dogv(g0, plane, w, layer, r - 1, c + 1) + dogv(g0, plane, w, layer, r - 1, c - 1)) * cross_scale;
            const float dxs = (dogv(g0, plane, w, layer + 1, r, c + 1) - dogv(g0, plane, w, layer + 1, r, c - 1) -
                               dogv(g0, plane, w, layer - 1, r, c + 1) + dogv(g0, plane, w, layer - 1, r, c - 1)) * cross_scale;
            const float dys = (dogv(g0, plane, w, layer + 1, r + 1, c) - dogv(g0, plane, w, layer + 1, r - 1, c) -
                               dogv(g0, plane, w, layer - 1, r + 1, c) + dogv(g0, plane, w, layer - 1, r - 1, c)) * cross_scale;
            float A[3][3] = {{dxx, dxy, dxs}, {dxy, dyy, dys}, {dxs, dys, dss}};
            float X[3] = {0.f, 0.f, 0.f};
            if (!solve3(A, dD, X)) { X[0] = X[1] = X[2] = 0.f; }
            xi = -X[2]; xr = -X[1]; xc = -X[0];
            if (fabsf(xi) < 0.5f && fabsf(xr) < 0.5f && fabsf(xc) < 0.5f) break;
            if (fabsf(xi) > 7e8f || fabsf(xr) > 7e8f || fabsf(xc) > 7e8f) { alive = false; break; }
            c += __float2int_rn(xc); r += __float2int_rn(xr); layer += __float2int_rn(xi);
            if (layer < 1 || layer > kLayers || c < kBorder || c >= w - kBorder || r < kBorder || r >= h - kBorder) { alive = false; break; }
        }
        if (alive && i < 5) {
            const float d0 = (dogv(g0, plane, w, layer, r, c + 1) - dogv(g0, plane, w, layer, r, c - 1)) * deriv_scale;
            const float d1 = (dogv(g0, plane, w, layer, r + 1, c) - dogv(g0, plane, w, layer, r - 1, c)) * deriv_scale;
            const float d2 = (dogv(g0, plane, w, layer + 1, r, c) - dogv(g0, plane, w, layer - 1, r, c)) * deriv_scale;
            const float t = d0 * xc + d1 * xr + d2 * xi;
            const float v = dogv(g0, plane, w, layer, r, c);
            contr = v * img_scale + t * 0.5f;
            if (fabsf(contr) * kLayers >= kContrastThr) {
                const float v2 = v * 2.f;
                const float dxx = (dogv(g0, plane, w, layer, r, c + 1) + dogv(g0, plane, w, layer, r, c - 1) - v2) * second_scale;
                const float dyy = (dogv(g0, plane, w, layer, r + 1, c) + dogv(g0, plane, w, layer, r - 1, c) - v2) * second_scale;
                const float dxy = (dogv(g0, plane, w, layer, r + 1, c + 1) - dogv(g0, plane, w, layer, r + 1, c - 1) -
                                   dogv(g0, plane, w, layer, r - 1, c + 1) + dogv(g0, plane, w, layer, r - 1, c - 1)) * cross_scale;
                const float tr = dxx + dyy, det = dxx * dyy - dxy * dxy;
                if (det > 0.f && tr * tr * kEdgeThr < (kEdgeThr + 1.f) * (kEdgeThr + 1.f) * det) ok = 1;
            }
        }
    }
    ok = __shfl_sync(0xffffffffu, ok, 0);
    if (!ok) continue;
    layer = __shfl_sync(0xffffffffu, layer, 0); r = __shfl_sync(0xffffffffu, r, 0); c = __shfl_sync(0xffffffffu, c, 0);
    xi = __shfl_sync(0xffffffffu, xi, 0); xr = __shfl_sync(0xffffffffu, xr, 0); xc = __shfl_sync(0xffffffffu, xc, 0);
    contr = __shfl_sync(0xffffffffu, contr, 0);
    const float oct_scale = (float)(1 << o);
    SiftKp kp;
    kp.x = (c + xc) * oct_scale; kp.y = (r + xr) * oct_scale;
    kp.octave = o + (layer << 8) + (__float2int_rn((xi + 0.5f) * 255.f) << 16);
    kp.size = kSigma * powf(2.f, (layer + xi) / kLayers) * oct_scale * 2.f;
    kp.response = fabsf(contr);

    // ---- calcOrientationHist on the Gaussian image of that layer ---------------------------------
    const float scl_octv = kp.size * 0.5f / oct_scale;
    const int radius = __float2int_rn(4.5f * scl_octv);
    const float sig = 1.5f * scl_octv;
    const float expf_scale = -1.f / (2.f * sig * sig);
    const float* img = g0 + (size_t)layer * plane;
    float* hist = hist_s[wl];
    for (int i = lane; i < 40; i += 32) hist[i] = 0.f;
    __syncwarp();
    const int side = 2 * radius + 1;
    for (int k = lane; k < side * side; k += 32) {
        const int i = k / side - radius, j = k - (k / side) * side - radius;
        const int y = r + i, x = c + j;
        if (y <= 0 || y >= h - 1 || x <= 0 || x >= w - 1) continue;
        const float dx = img[(size_t)y * w + x + 1] - img[(size_t)y * w + x - 1];
        const float dy = img[(size_t)(y - 1) * w + x] - img[(size_t)(y + 1) * w + x];
        const float wgt = expf((i * i + j * j) * expf_scale);
        const float ori = atan2_deg(dy, dx), mag = sqrtf(dx * dx + dy * dy);
        int bin = __float2int_rn((36.f / 360.f) * ori);
        if (bin >= 36) bin -= 36;
        if (bin < 0) bin += 36;
        atomicAdd(&hist[2 + bin], wgt * mag);
    }
    __syncwarp();
    if (lane == 0) { hist[0] = hist[2 + 34]; hist[1] = hist[2 + 35]; hist[38] = hist[2]; hist[39] = hist[3]; }
    __syncwarp();
    float sm0 = 0.f, sm1 = 0.f;                 // smoothed bins lane and lane+32
    {
        const int b = lane;
        sm0 = (hist[b] + hist[b + 4]) * (1.f / 16.f) + (hist[b + 1] + hist[b + 3]) * (4.f / 16.f) + hist[b + 2] * (6.f / 16.f);
        if (lane < 4) { const int b2 = lane + 32; sm1 = (hist[b2] + hist[b2 + 4]) * (1.f / 16.f) + (hist[b2 + 1] + hist[b2 + 3]) * (4.f / 16.f) + hist[b2 + 2] * (6.f / 16.f); }
    }
    __syncwarp();
    hist[lane] = sm0;
    if (lane < 4) hist[lane + 32] = sm1;
    __syncwarp();
    float mx = fmaxf(sm0, lane < 4 ? sm1 : 0.f);
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, s));
    const float mag_thr = mx * 0.8f;
    for (int j = lane; j < 36; j += 32) {
        const int l = j > 0 ? j - 1 : 35, r2 = j < 35 ? j + 1 : 0;
        const float hj = hist[j], hl = hist[l], hr = hist[r2];
        if (hj > hl && hj > hr && hj >= mag_thr) {
            float bin = j + 0.5f * (hl - hr) / (hl - 2.f * hj + hr);
            bin = bin < 0.f ? 36.f + bin : (bin >= 36.f ? bin - 36.f : bin);
            SiftKp k2 = kp;
            k2.angle = 360.f - (360.f / 36.f) * bin;
            if (fabsf(k2.angle - 360.f) < 1.1920929e-7f) k2.angle = 0.f;
            const int pos = atomicAdd(nkp, 1);
            if (pos < kcap) kps[pos] = k2;
        }
    }
    }
}

// ---------------------------------------------------------------- ordering / duplicates / retainBest
__global__ void __launch_bounds__(256)
sift_keys_kernel(const SiftKp* __restrict__ kps, const int* __restrict__ nkp, int kcap, unsigned long long* __restrict__ keys,
                 int* __restrict__ idx) {
    const int n = min(*nkp, kcap);
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= kcap) return;
    idx[i] = i;
    if (i >= n) { keys[i] = ~0ull; return; }
    // KeyPoint_LessThan orders by x then y (then size desc, angle, ...): x | y as sortable float bits
    auto ord = [](float f) { unsigned u = __float_as_uint(f); return (u & 0x80000000u) ? ~u : (u | 0x80000000u); };
    keys[i] = ((unsigned long long)ord(kps[i].x) << 32) | (unsigned long long)ord(kps[i].y);
}

// after sorting by (x, y): drop a keypoint when an earlier one in its (x, y) run has the same size and
// angle (KeyPointsFilter::removeDuplicatedSorted); write the response keys of the survivors
__global__ void __launch_bounds__(256)
sift_dedupe_kernel(const SiftKp* __restrict__ kps, const int* __restrict__ nkp, int kcap, const unsigned long long* __restrict__ skeys,
                   const int* __restrict__ sidx, unsigned int* __restrict__ rkeys, uint8_t* __restrict__ alive) {
    const int n = min(*nkp, kcap);
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= kcap) return;
    if (i >= n) { rkeys[i] = 0u; alive[i] = 0; return; }
    const SiftKp a = kps[sidx[i]];
    bool dup = false;
    for (int j = i - 1; j >= 0 && j >= i - 16 && skeys[j] == skeys[i]; --j) {
        const SiftKp b = kps[sidx[j]];
        if (b.size == a.size && b.angle == a.angle) { dup = true; break; }
    }
    alive[i] = dup ? 0 : 1;
    rkeys[i] = dup ? 0u : __float_as_uint(a.response);          // responses are >= 0: bit order == value order
}

// threshold = nfeatures-th largest response among the survivors (ties kept), then compaction in (x, y)
// order with the octave -1 rescale (x0.5) and the reference's relative-size filter.  Single CTA.
__global__ void __launch_bounds__(1024)
sift_select_kernel(const SiftKp* __restrict__ kps, const int* __restrict__ nkp, int kcap, const int* __restrict__ sidx,
                   const uint8_t* __restrict__ alive, const unsigned int* __restrict__ rsorted /* descending */, int nfeatures,
                   float max_size, SiftKp* __restrict__ out, int* __restrict__ nout, int max_out) {
    __shared__ int wsum[32];
    __shared__ int s_base;
    const int n = min(*nkp, kcap);
    const unsigned thr = (nfeatures > 0 && n > nfeatures) ? rsorted[nfeatures - 1] : 0u;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_base = 0;
    __syncthreads();
    for (int base = 0; base < n; base += 1024) {
        const int i = base + threadIdx.x;
        bool keep = false;
        SiftKp k;
        if (i < n && alive[i]) {
            k = kps[sidx[i]];
            keep = __float_as_uint(k.response) >= thr && thr != 0u ? true : (thr == 0u);
            if (keep) {
                // firstOctave = -1: scale back to input-image coordinates
                k.octave = (k.octave & ~255) | ((k.octave - 1) & 255);
                k.x *= 0.5f; k.y *= 0.5f; k.size *= 0.5f;
                if (max_size > 0.f && !(k.size < max_size)) keep = false;          // :290-309
            }
        }
        const unsigned ball = __ballot_sync(0xffffffffu, keep);
        if (lane == 0) wsum[wid] = __popc(ball);
        __syncthreads();
        int off = s_base;
        for (int w2 = 0; w2 < wid; ++w2) off += wsum[w2];
        if (keep) {
            const int pos = off + __popc(ball & ((1u << lane) - 1u));
            if (pos < max_out) out[pos] = k;
        }
        __syncthreads();
        if (threadIdx.x == 0) { int t = 0; for (int w2 = 0; w2 < 32; ++w2) t += wsum[w2]; s_base += t; }
        __syncthreads();
    }
    if (threadIdx.x == 0) *nout = min(s_base, max_out);
}

// ---------------------------------------------------------------- descriptor, one CTA of 128 threads per keypoint
__global__ void __launch_bounds__(128)
sift_descriptor_kernel(const float* __restrict__ pyr, SiftOctaves O, const SiftKp* __restrict__ kps, const int* __restrict__ nkp,
                       int max_kp, uint8_t* __restrict__ desc) {
    constexpr int d = 4, nb = 8;
    __shared__ float hist[(d + 2) * (d + 2) * (nb + 2)];
    __shared__ float dst[d * d * nb];
    __shared__ float red[4];
    const int n = min(*nkp, max_kp);
    const int ki = blockIdx.x;
    if (ki >= n) return;
    const SiftKp kp = kps[ki];
    // unpackOctave
    int octave = kp.octave & 255;
    const int layer = (kp.octave >> 8) & 255;
    octave = octave < 128 ? octave : (-128 | octave);
    const float scale = octave >= 0 ? 1.f / (float)(1 << octave) : (float)(1 << -octave);
    const int o = octave + 1;                                  // octave index in the pyramid (firstOctave = -1)
    const int w = O.w[o], h = O.h[o];
    const float* img = pyr + O.off[o] + (size_t)layer * w * h;
    const float size = kp.size * scale;
    const float px = kp.x * scale, py = kp.y * scale;
    float ori = 360.f - kp.angle;
    if (fabsf(ori - 360.f) < 1.1920929e-7f) ori = 0.f;
    const float scl = size * 0.5f;
    const int ptx = __float2int_rn(px), pty = __float2int_rn(py);
    float cos_t = cosf(ori * (float)(3.14159265358979323846 / 180.0)), sin_t = sinf(ori * (float)(3.14159265358979323846 / 180.0));
    const float bins_per_rad = nb / 360.f, exp_scale = -1.f / (d * d * 0.5f), hist_width = 3.f * scl;
    int radius = __float2int_rn(hist_width * 1.4142135623730951f * (d + 1) * 0.5f);
    radius = min(radius, (int)sqrt((double)w * w + (double)h * h));
    cos_t /= hist_width; sin_t /= hist_width;
    for (int i = threadIdx.x; i < (d + 2) * (d + 2) * (nb + 2); i += 128) hist[i] = 0.f;
    __syncthreads();
    const int side = 2 * radius + 1;
    for (int k = threadIdx.x; k < side * side; k += 128) {
        const int i = k / side - radius, j = k - (k / side) * side - radius;
        const float c_rot = j * cos_t - i * sin_t, r_rot = j * sin_t + i * cos_t;
        float rbin = r_rot + d / 2 - 0.5f, cbin = c_rot + d / 2 - 0.5f;
        const int r = pty + i, c = ptx + j;
        if (rbin > -1 && rbin < d && cbin > -1 && cbin < d && r > 0 && r < h - 1 && c > 0 && c < w - 1) {
            const float dx = img[(size_t)r * w + c + 1] - img[(size_t)r * w + c - 1];
            const float dy = img[(size_t)(r - 1) * w + c] - img[(size_t)(r + 1) * w + c];
            const float wgt = expf((c_rot * c_rot + r_rot * r_rot) * exp_scale);
            float obin = (atan2_deg(dy, dx) - ori) * bins_per_rad;
            const float mag = sqrtf(dx * dx + dy * dy) * wgt;
            const int r0 = (int)floorf(rbin), c0 = (int)floorf(cbin);
            int o0 = (int)floorf(obin);
            rbin -= r0; cbin -= c0; obin -= o0;
            if (o0 < 0) o0 += nb;
            if (o0 >= nb) o0 -= nb;
            const float v_r1 = mag * rbin, v_r0 = mag - v_r1;
            const float v_rc11 = v_r1 * cbin, v_rc10 = v_r1 - v_rc11;
            const float v_rc01 = v_r0 * cbin, v_rc00 = v_r0 - v_rc01;
            const float v_rco111 = v_rc11 * obin, v_rco110 = v_rc11 - v_rco111;
            const float v_rco101 = v_rc10 * obin, v_rco100 = v_rc10 - v_rco101;
            const float v_rco011 = v_rc01 * obin, v_rco010 = v_rc01 - v_rco011;
            const float v_rco001 = v_rc00 * obin, v_rco000 = v_rc00 - v_rco001;
            const int idx = ((r0 + 1) * (d + 2) + c0 + 1) * (nb + 2) + o0;
            atomicAdd(&hist[idx], v_rco000);
            atomicAdd(&hist[idx + 1], v_rco001);
            atomicAdd(&hist[idx + (nb + 2)], v_rco010);
            atomicAdd(&hist[idx + (nb + 3)], v_rco011);
            atomicAdd(&hist[idx + (d + 2) * (nb + 2)], v_rco100);
            atomicAdd(&hist[idx + (d + 2) * (nb + 2) + 1], v_rco101);
            atomicAdd(&hist[idx + (d + 3) * (nb + 2)], v_rco110);
            atomicAdd(&hist[idx + (d + 3) * (nb + 2) + 1], v_rco111);
        }
    }
    __syncthreads();
    // finalize: fold the circular orientation bins, gather the 4x4x8 core
    {
        const int t = threadIdx.x;                 // 128 = d*d*nb outputs
        const int i = t / (d * nb), j = (t / nb) % d, k = t % nb;
        const int idx = ((i + 1) * (d + 2) + (j + 1)) * (nb + 2);
        float v = hist[idx + k];
        if (k == 0) v += hist[idx + nb];
        if (k == 1) v += hist[idx + nb + 1];
        dst[t] = v;
    }
    __syncthreads();
    auto block_sum = [&](float v) {
#pragma unroll
        for (int s = 16; s > 0; s >>= 1) v += __shfl_xor_sync(0xffffffffu, v, s);
        __syncthreads();
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
        __syncthreads();
        return red[0] + red[1] + red[2] + red[3];
    };
    const float v0 = dst[threadIdx.x];
    const float nrm2 = block_sum(v0 * v0);
    const float thr = sqrtf(nrm2) * 0.2f;
    const float v1 = fminf(v0, thr);
    float nrm = block_sum(v1 * v1);
    nrm = 512.f / fmaxf(sqrtf(nrm), 1.1920929e-7f);
    const int q = __float2int_rn(v1 * nrm);
    desc[(size_t)ki * 128 + threadIdx.x] = (uint8_t)min(255, max(0, q));
}

}  // namespace

// ------------------------------------------------------------------------------------------------
static size_t al256(size_t v) { return (v + 255) & ~(size_t)255; }

static void gaussian_kernel(double sigma, int* radius, float* out) {
    int ksize = (int)std::lrint(sigma * 4 * 2 + 1) | 1;                 // cvRound(sigma*4*2 + 1) | 1 (float images)
    int R = ksize / 2;
    if (R > kMaxRadius) R = kMaxRadius;
    std::vector<double> k(2 * R + 1);
    double sum = 0;
    for (int i = -R; i <= R; ++i) { k[i + R] = std::exp(-0.5 * i * i / (sigma * sigma)); sum += k[i + R]; }
    for (int i = 0; i <= 2 * R; ++i) out[i] = (float)(k[i] / sum);
    *radius = R;
}

SiftPlan* sift_plan_create(int w, int h, double size_ratio, int max_keypoints, std::string* err) {
    SiftPlan* P = new SiftPlan();
    P->w = w; P->h = h; P->max_kp = max_keypoints;
    P->max_size = size_ratio > 0.0 ? (float)(size_ratio * h) : 0.f;
    SiftOctaves& O = *new SiftOctaves();
    P->octaves = &O;
    const int bw = 2 * w, bh = 2 * h;
    int nOct = (int)std::lrint(std::log((double)std::min(bw, bh)) / std::log(2.0) - 2.0) + 1;     // - firstOctave (= -1)
    if (nOct > kSiftMaxOctaves) nOct = kSiftMaxOctaves;
    if (nOct < 1) nOct = 1;
    O.n = nOct;
    size_t off = 0;
    int cw = bw, ch = bh;
    for (int o = 0; o < nOct; ++o) {
        O.w[o] = cw; O.h[o] = ch; O.off[o] = off;
        off += (size_t)kGauss * cw * ch;
        cw /= 2; ch /= 2;
        if (cw < 1 || ch < 1) { O.n = o + 1; break; }
    }
    P->pyr_floats = off;
    P->cand_cap = (int)al256((size_t)bw * bh / 16 + 65536);
    P->kp_cap = 1 << 18;
    // Gaussian kernels: initial blur sqrt(sigma^2 - (2*0.5)^2), then the incremental sigmas of the octave
    float hk[kGauss + 1][2 * kMaxRadius + 1] = {};
    int hr[kGauss + 1] = {};
    const double sigma = 1.2;
    double sig_diff = std::sqrt(std::max(sigma * sigma - 4.0 * 0.5 * 0.5, 0.01));
    gaussian_kernel(sig_diff, &hr[0], hk[0]);
    const double k = std::pow(2.0, 1.0 / kLayers);
    for (int i = 1; i < kGauss; ++i) {
        const double sp = std::pow(k, (double)(i - 1)) * sigma, st = sp * k;
        gaussian_kernel(std::sqrt(st * st - sp * sp), &hr[i], hk[i]);
    }
    cudaMemcpyToSymbol(c_gk, hk, sizeof(hk));
    cudaMemcpyToSymbol(c_gr, hr, sizeof(hr));
    for (int i = 0; i <= kGauss; ++i) P->radii[i] = hr[i];
    size_t t1 = 0, t2 = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, t1, (const unsigned long long*)nullptr, (unsigned long long*)nullptr, (const int*)nullptr,
                                    (int*)nullptr, P->kp_cap);
    cub::DeviceRadixSort::SortKeysDescending(nullptr, t2, (const unsigned int*)nullptr, (unsigned int*)nullptr, P->kp_cap);
    P->cub_bytes = t1 > t2 ? t1 : t2;
    const size_t bytes = al256(sizeof(float) * P->pyr_floats) + al256(8 * (size_t)P->cand_cap) + al256(sizeof(SiftKp) * P->kp_cap) +
                         2 * al256(8 * (size_t)P->kp_cap) + 2 * al256(4 * (size_t)P->kp_cap) + 2 * al256(4 * (size_t)P->kp_cap) +
                         al256(P->kp_cap) + al256(256) + al256(P->cub_bytes);
    if (cudaMalloc(&P->mem, bytes) != cudaSuccess) { if (err) *err = "cudaMalloc(SIFT workspace) failed"; delete &O; delete P; return nullptr; }
    char* b = (char*)P->mem;
    P->pyr = (float*)b; b += al256(sizeof(float) * P->pyr_floats);
    P->cand = (unsigned long long*)b; b += al256(8 * (size_t)P->cand_cap);
    P->kps = b; b += al256(sizeof(SiftKp) * P->kp_cap);
    P->keys = (unsigned long long*)b; b += al256(8 * (size_t)P->kp_cap);
    P->keys_sorted = (unsigned long long*)b; b += al256(8 * (size_t)P->kp_cap);
    P->idx = (int*)b; b += al256(4 * (size_t)P->kp_cap);
    P->idx_sorted = (int*)b; b += al256(4 * (size_t)P->kp_cap);
    P->rkeys = (unsigned int*)b; b += al256(4 * (size_t)P->kp_cap);
    P->rkeys_sorted = (unsigned int*)b; b += al256(4 * (size_t)P->kp_cap);
    P->alive = (uint8_t*)b; b += al256(P->kp_cap);
    P->counters = (int*)b; b += al256(256);
    P->cub_temp = b;
    return P;
}

void sift_plan_destroy(SiftPlan* P) {
    if (!P) return;
    for (auto& a : P->aux) if (a) cudaStreamDestroy(a);
    for (auto& e : P->ev_g3) if (e) cudaEventDestroy(e);
    for (auto& e : P->ev_join) if (e) cudaEventDestroy(e);
    if (P->mem) cudaFree(P->mem);
    delete (SiftOctaves*)P->octaves;
    delete P;
}

static void launch_sift_body(SiftPlan* P, const uint8_t* gray, OrbKeypoint* kps_out, uint8_t* desc, int* count, cudaStream_t st);

void launch_sift(SiftPlan* P, const uint8_t* gray, OrbKeypoint* kps_out, uint8_t* desc, int* count, cudaStream_t st) {
    // ~120 small dependent launches per frame: replayed as one CUDA graph from the third call with the same buffers on
    const unsigned long long key[5] = {(unsigned long long)gray, (unsigned long long)kps_out, (unsigned long long)desc,
                                       (unsigned long long)count, (unsigned long long)st};
    run_graphed(P->graphs, key, st, [&] { launch_sift_body(P, gray, kps_out, desc, count, st); });
}

static void launch_sift_body(SiftPlan* P, const uint8_t* gray, OrbKeypoint* kps_out, uint8_t* desc, int* count, cudaStream_t st) {
    SiftOctaves& O = *(SiftOctaves*)P->octaves;
    const int max_smem = (int)(sizeof(float) * ((GBY + 2 * kMaxRadius) * (GBX + 2 * kMaxRadius) + (GBY + 2 * kMaxRadius) * GBX));
    static PerDeviceOnce once;
    once.run([&] { cudaFuncSetAttribute(sift_blur_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem); });
    const int* hr = P->radii;
    auto blur = [&](const float* src, float* dst, int w, int h, int ki, cudaStream_t st) {
        const int R = hr[ki];
        switch (R) {                       // the radii of SIFT's sigmas; anything else takes the generic kernel
            case 3: launch_blur_t<3>(src, dst, w, h, ki, st); return;
            case 4: launch_blur_t<4>(src, dst, w, h, ki, st); return;
            case 5: launch_blur_t<5>(src, dst, w, h, ki, st); return;
            case 6: launch_blur_t<6>(src, dst, w, h, ki, st); return;
            case 8: launch_blur_t<8>(src, dst, w, h, ki, st); return;
            case 10: launch_blur_t<10>(src, dst, w, h, ki, st); return;
            default: break;
        }
        const int smem = (int)(sizeof(float) * ((GBY + 2 * R) * (GBX + 2 * R) + (GBY + 2 * R) * GBX));
        sift_blur_kernel<<<dim3((w + GBX - 1) / GBX, (h + GBY - 1) / GBY), 256, smem, st>>>(src, dst, w, h, ki);
    };
    int launches = 3;
    cudaMemsetAsync(P->counters, 0, 256, st);
    cudaMemsetAsync(count, 0, sizeof(int), st);
    // base image: upsample into the Gaussian-1 slot of octave 0 (scratch), blur into Gaussian 0
    float* g0 = P->pyr + O.off[0];
    float* scratch = g0 + (size_t)O.w[0] * O.h[0];
    sift_upsample_kernel<<<dim3((P->w + 255) / 256, P->h), 256, 0, st>>>(gray, P->w, P->h, scratch);
    blur(scratch, g0, O.w[0], O.h[0], 0, st);
    const int threshold = (int)std::floor(0.5 * 0.04 / kLayers * 255.0);
    // Octave o + 1 starts from Gaussian[kLayers] of octave o, so it does not have to wait for the last two blurs and the
    // extrema pass of octave o: octaves >= 1 alternate between two auxiliary streams (fork / join by events; inside a
    // graph capture these become parallel branches).  The small octaves are ~40 launches of a few CTAs each, about
    // 0.5 ms of pure latency per 4K frame when they run behind octave 0 instead of beside it.
    if (!P->aux[0]) {
        // highest priority: their few CTAs are dispatched ahead of the thousands queued by the octave-0 kernels
        int prio_lo = 0, prio_hi = 0;
        cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
        for (auto& a : P->aux) cudaStreamCreateWithPriority(&a, cudaStreamNonBlocking, prio_hi);
        for (auto& e : P->ev_g3) cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
        for (auto& e : P->ev_join) cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
    }
    bool used[2] = {false, false};
    for (int o = 0; o < O.n; ++o) {
        const int w = O.w[o], h = O.h[o];
        const size_t plane = (size_t)w * h;
        float* g = P->pyr + O.off[o];
        const int lane = (o - 1) & 1;
        cudaStream_t q = o > 0 ? P->aux[lane] : st;
        if (o > 0) {
            cudaStreamWaitEvent(q, P->ev_g3[o - 1], 0);
            used[lane] = true;
            const float* src = P->pyr + O.off[o - 1] + (size_t)kLayers * O.w[o - 1] * O.h[o - 1];
            sift_decimate_kernel<<<dim3((w + 255) / 256, h), 256, 0, q>>>(src, O.w[o - 1], g, w, h);
            ++launches;
        }
        for (int i = 1; i < kGauss; ++i) {
            blur(g + (size_t)(i - 1) * plane, g + (size_t)i * plane, w, h, i, q);
            ++launches;
            if (i == kLayers && o + 1 < O.n) cudaEventRecord(P->ev_g3[o], q);
        }
        if (w > 2 * kBorder && h > 2 * kBorder) {
            sift_extrema_tile_kernel<<<dim3((w - 2 * kBorder + EXW - 1) / EXW, (h - 2 * kBorder + EXH - 1) / EXH), 256, 0, q>>>(
                P->pyr, O, o, threshold, P->cand, P->counters + 0, P->cand_cap);
            ++launches;
        }
    }
    for (int k = 0; k < 2; ++k)
        if (used[k]) { cudaEventRecord(P->ev_join[k], P->aux[k]); cudaStreamWaitEvent(st, P->ev_join[k], 0); }
    SiftKp* kps = (SiftKp*)P->kps;
    sift_refine_kernel<<<std::min((P->cand_cap + 3) / 4, 148 * 16), 128, 0, st>>>(P->pyr, O, P->cand, P->counters + 0, P->cand_cap, kps, P->counters + 1,
                                                             P->kp_cap);
    sift_keys_kernel<<<(P->kp_cap + 255) / 256, 256, 0, st>>>(kps, P->counters + 1, P->kp_cap, P->keys, P->idx);
    size_t temp = P->cub_bytes;
    cub::DeviceRadixSort::SortPairs(P->cub_temp, temp, (const unsigned long long*)P->keys, P->keys_sorted, (const int*)P->idx,
                                    P->idx_sorted, P->kp_cap, 0, 64, st);
    sift_dedupe_kernel<<<(P->kp_cap + 255) / 256, 256, 0, st>>>(kps, P->counters + 1, P->kp_cap, P->keys_sorted, P->idx_sorted,
                                                               P->rkeys, P->alive);
    temp = P->cub_bytes;
    cub::DeviceRadixSort::SortKeysDescending(P->cub_temp, temp, (const unsigned int*)P->rkeys, P->rkeys_sorted, P->kp_cap, 0, 32, st);
    sift_select_kernel<<<1, 1024, 0, st>>>(kps, P->counters + 1, P->kp_cap, P->idx_sorted, P->alive, P->rkeys_sorted, 2500,
                                          P->max_size, (SiftKp*)kps_out, count, P->max_kp);
    sift_descriptor_kernel<<<P->max_kp, 128, 0, st>>>(P->pyr, O, (const SiftKp*)kps_out, count, P->max_kp, desc);
    count_launch(launches + 6);
}

}  // namespace vstabk
