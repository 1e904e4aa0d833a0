// K15 YUV 4:2:0 <-> BGR: the frame formats of video decoders and encoders (NV12 from NVDEC, yuv420p / I420 from ffmpeg)
// converted on the device, so that 1.5 instead of 3 bytes per pixel cross the host link.  Bit-exact with OpenCV 4.x
// (BT.601 limited range, 20-bit fixed point, int32 arithmetic):
//   cvtColor(COLOR_YUV2BGR_NV12 / COLOR_YUV2BGR_I420): the chroma sample of a 2x2 block serves its four pixels;
//   cvtColor(COLOR_BGR2YUV_I420): luma of every pixel, chroma of the TOP-LEFT pixel of each 2x2 block (no averaging).
// NV12 output is I420's chroma interleaved U,V.  One kernel per direction serves both formats: the chroma planes are
// (pointer, row step, sample step) with a sample step of 2 for NV12's interleaved plane and 1 for I420's.
//
// HBM-bound (4.5 bytes per pixel either way).  A thread owns 2 rows x 8 pixels = one row of 4 chroma samples: with
// aligned planes it moves them with 8-byte (Y, NV12 chroma, BGR) and 4-byte (I420 chroma) loads and stores; caller
// memory whose pointers or steps are not aligned takes the byte path, as do the last columns of a row when cols % 8 != 0.
#include "kernels.h"

namespace vstabk {

namespace {

constexpr int kYuvShift = 20;
constexpr int kYuvHalf = 1 << (kYuvShift - 1);
// YUV -> BGR (OpenCV's ITUR_BT_601_CY, _CVR, _CVG, _CUG, _CUB)
constexpr int kCY = 1220542, kCVR = 1673527, kCVG = -852492, kCUG = -409993, kCUB = 2116026;
// BGR -> YUV (OpenCV's ITUR_BT_601_CRY, _CGY, _CBY, _CRU, _CGU, _CBU, _CGV, _CBV; CRV == CBU)
constexpr int kRY = 269484, kGY = 528482, kBY = 102760;
constexpr int kRU = -155188, kGU = -305135, kBU = 460324;
constexpr int kRV = 460324, kGV = -385875, kBV = -74448;
constexpr int kYuvThreadsX = 32, kYuvThreadsY = 4;

__device__ __forceinline__ unsigned clip8(int v) { return (unsigned)min(max(v, 0), 255); }

// chroma terms of one sample, shared by the four pixels of its block
struct Chroma { int b, g, r; };
__device__ __forceinline__ Chroma chroma_terms(unsigned U, unsigned V) {
    const int u = (int)U - 128, v = (int)V - 128;
    return {kYuvHalf + kCUB * u, kYuvHalf + kCVG * v + kCUG * u, kYuvHalf + kCVR * v};
}
// B | G << 8 | R << 16 of one pixel
__device__ __forceinline__ unsigned yuv_pixel(unsigned Y, const Chroma& c) {
    const int y = max((int)Y - 16, 0) * kCY;
    return clip8((y + c.b) >> kYuvShift) | (clip8((y + c.g) >> kYuvShift) << 8) | (clip8((y + c.r) >> kYuvShift) << 16);
}
// every intermediate is within [0, 2^28): no clipping needed for in-range bytes
__device__ __forceinline__ unsigned luma_of(int b, int g, int r) {
    return (unsigned)((kRY * r + kGY * g + kBY * b + kYuvHalf + (16 << kYuvShift)) >> kYuvShift);
}
__device__ __forceinline__ unsigned cb_of(int b, int g, int r) {
    return (unsigned)((kRU * r + kGU * g + kBU * b + kYuvHalf + (128 << kYuvShift)) >> kYuvShift);
}
__device__ __forceinline__ unsigned cr_of(int b, int g, int r) {
    return (unsigned)((kRV * r + kGV * g + kBV * b + kYuvHalf + (128 << kYuvShift)) >> kYuvShift);
}
__device__ __forceinline__ unsigned byte_of(const unsigned (&w)[6], int i) { return (w[i >> 2] >> (8 * (i & 3))) & 0xffu; }

template <bool kVec>
__global__ void __launch_bounds__(kYuvThreadsX * kYuvThreadsY)
yuv420_to_bgr_kernel(const uint8_t* __restrict__ yuv, YuvPlanes L, size_t yuv_frame_stride, int rows, int cols,
                     uint8_t* __restrict__ bgr, size_t pitch, size_t frame_stride) {
    const int x0 = 8 * (blockIdx.x * kYuvThreadsX + threadIdx.x);
    const int cy = blockIdx.y * kYuvThreadsY + threadIdx.y;          // chroma row = rows 2cy, 2cy + 1
    if (x0 >= cols || 2 * cy >= rows) return;
    const uint8_t* f = yuv + (size_t)blockIdx.z * yuv_frame_stride;
    const uint8_t* y0 = f + L.off_y + (size_t)(2 * cy) * L.step_y + x0;
    const uint8_t* y1 = y0 + L.step_y;
    const uint8_t* up = f + L.off_u + (size_t)cy * L.step_u + (size_t)(x0 >> 1) * L.cstep;
    const uint8_t* vp = f + L.off_v + (size_t)cy * L.step_v + (size_t)(x0 >> 1) * L.cstep;
    uint8_t* o0 = bgr + (size_t)blockIdx.z * frame_stride + (size_t)(2 * cy) * pitch + (size_t)x0 * 3;
    uint8_t* o1 = o0 + pitch;
    if (kVec && x0 + 8 <= cols) {
        const uint2 a = __ldg(reinterpret_cast<const uint2*>(y0));
        const uint2 b = __ldg(reinterpret_cast<const uint2*>(y1));
        unsigned uu, vv;                                             // 4 U / 4 V bytes
        if (L.cstep == 2) {
            const uint2 c = __ldg(reinterpret_cast<const uint2*>(up));   // U0 V0 U1 V1 | U2 V2 U3 V3
            uu = __byte_perm(c.x, c.y, 0x6420);
            vv = __byte_perm(c.x, c.y, 0x7531);
        } else {
            uu = __ldg(reinterpret_cast<const unsigned*>(up));
            vv = __ldg(reinterpret_cast<const unsigned*>(vp));
        }
        const unsigned yw[2][2] = {{a.x, a.y}, {b.x, b.y}};
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            unsigned w[6] = {0, 0, 0, 0, 0, 0};
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const Chroma c = chroma_terms((uu >> (8 * (i >> 1))) & 0xffu, (vv >> (8 * (i >> 1))) & 0xffu);
                const unsigned px = yuv_pixel((yw[r][i >> 2] >> (8 * (i & 3))) & 0xffu, c);
#pragma unroll
                for (int ch = 0; ch < 3; ++ch) {
                    const int bi = 3 * i + ch;
                    w[bi >> 2] |= ((px >> (8 * ch)) & 0xffu) << (8 * (bi & 3));
                }
            }
            uint2* o = reinterpret_cast<uint2*>(r ? o1 : o0);
            o[0] = make_uint2(w[0], w[1]);
            o[1] = make_uint2(w[2], w[3]);
            o[2] = make_uint2(w[4], w[5]);
        }
        return;
    }
    const int n = min(8, cols - x0);                                 // even: cols is even
    for (int i = 0; i < n; i += 2) {
        const Chroma c = chroma_terms(up[(i >> 1) * L.cstep], vp[(i >> 1) * L.cstep]);
#pragma unroll
        for (int d = 0; d < 2; ++d) {
            const unsigned p0 = yuv_pixel(y0[i + d], c), p1 = yuv_pixel(y1[i + d], c);
            uint8_t* q0 = o0 + 3 * (i + d);
            uint8_t* q1 = o1 + 3 * (i + d);
            q0[0] = (uint8_t)p0; q0[1] = (uint8_t)(p0 >> 8); q0[2] = (uint8_t)(p0 >> 16);
            q1[0] = (uint8_t)p1; q1[1] = (uint8_t)(p1 >> 8); q1[2] = (uint8_t)(p1 >> 16);
        }
    }
}

template <bool kVec>
__global__ void __launch_bounds__(kYuvThreadsX * kYuvThreadsY)
bgr_to_yuv420_kernel(const uint8_t* __restrict__ bgr, size_t pitch, size_t frame_stride, int rows, int cols,
                     uint8_t* __restrict__ yuv, YuvPlanes L, size_t yuv_frame_stride) {
    const int x0 = 8 * (blockIdx.x * kYuvThreadsX + threadIdx.x);
    const int cy = blockIdx.y * kYuvThreadsY + threadIdx.y;
    if (x0 >= cols || 2 * cy >= rows) return;
    const uint8_t* s0 = bgr + (size_t)blockIdx.z * frame_stride + (size_t)(2 * cy) * pitch + (size_t)x0 * 3;
    const uint8_t* s1 = s0 + pitch;
    uint8_t* f = yuv + (size_t)blockIdx.z * yuv_frame_stride;
    uint8_t* y0 = f + L.off_y + (size_t)(2 * cy) * L.step_y + x0;
    uint8_t* y1 = y0 + L.step_y;
    uint8_t* up = f + L.off_u + (size_t)cy * L.step_u + (size_t)(x0 >> 1) * L.cstep;
    uint8_t* vp = f + L.off_v + (size_t)cy * L.step_v + (size_t)(x0 >> 1) * L.cstep;
    if (kVec && x0 + 8 <= cols) {
        unsigned w[2][6];
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            const uint2* s = reinterpret_cast<const uint2*>(r ? s1 : s0);
            const uint2 a = __ldg(s), b = __ldg(s + 1), c = __ldg(s + 2);
            w[r][0] = a.x; w[r][1] = a.y; w[r][2] = b.x; w[r][3] = b.y; w[r][4] = c.x; w[r][5] = c.y;
        }
        unsigned yo[2][2] = {{0, 0}, {0, 0}}, uu = 0, vv = 0;
#pragma unroll
        for (int r = 0; r < 2; ++r)
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int B = (int)byte_of(w[r], 3 * i), G = (int)byte_of(w[r], 3 * i + 1), R = (int)byte_of(w[r], 3 * i + 2);
                yo[r][i >> 2] |= luma_of(B, G, R) << (8 * (i & 3));
                if (r == 0 && !(i & 1)) {
                    uu |= cb_of(B, G, R) << (8 * (i >> 1));
                    vv |= cr_of(B, G, R) << (8 * (i >> 1));
                }
            }
        *reinterpret_cast<uint2*>(y0) = make_uint2(yo[0][0], yo[0][1]);
        *reinterpret_cast<uint2*>(y1) = make_uint2(yo[1][0], yo[1][1]);
        if (L.cstep == 2) {
            *reinterpret_cast<uint2*>(up) = make_uint2(__byte_perm(uu, vv, 0x5140), __byte_perm(uu, vv, 0x7362));
        } else {
            *reinterpret_cast<unsigned*>(up) = uu;
            *reinterpret_cast<unsigned*>(vp) = vv;
        }
        return;
    }
    const int n = min(8, cols - x0);
    for (int i = 0; i < n; ++i) {
        const uint8_t* p0 = s0 + 3 * i;
        const uint8_t* p1 = s1 + 3 * i;
        y0[i] = (uint8_t)luma_of(p0[0], p0[1], p0[2]);
        y1[i] = (uint8_t)luma_of(p1[0], p1[1], p1[2]);
        if (!(i & 1)) {
            up[(i >> 1) * L.cstep] = (uint8_t)cb_of(p0[0], p0[1], p0[2]);
            vp[(i >> 1) * L.cstep] = (uint8_t)cr_of(p0[0], p0[1], p0[2]);
        }
    }
}

inline bool aligned(uintptr_t v, uintptr_t a) { return (v & (a - 1)) == 0; }

// the word paths need 8-byte Y / NV12-chroma / BGR rows and 4-byte I420 chroma rows in every frame
bool vector_ok(const uint8_t* yuv, const YuvPlanes& L, size_t yuv_frame_stride, int cols, const uint8_t* bgr, size_t pitch,
               size_t frame_stride) {
    const uintptr_t f = (uintptr_t)yuv | yuv_frame_stride;
    const bool chroma = L.cstep == 2 ? aligned(f | L.off_u | L.step_u, 8)                 // NV12: U,V pairs in one plane
                                     : aligned(f | L.off_u | L.step_u | L.off_v | L.step_v, 4);
    return cols >= 8 && chroma && aligned(f | L.off_y | L.step_y, 8) && aligned((uintptr_t)bgr | pitch | frame_stride, 8);
}

dim3 yuv_grid(int rows, int cols, int nframes) {
    const int groups = (cols + 7) / 8;
    return dim3((groups + kYuvThreadsX - 1) / kYuvThreadsX, (rows / 2 + kYuvThreadsY - 1) / kYuvThreadsY, nframes);
}

}  // namespace

void launch_yuv420_to_bgr(const uint8_t* yuv, const YuvPlanes& L, size_t yuv_frame_stride, int nframes, int rows, int cols,
                          uint8_t* bgr, size_t pitch, size_t frame_stride, cudaStream_t st) {
    if (nframes <= 0) return;
    const dim3 grid = yuv_grid(rows, cols, nframes), block(kYuvThreadsX, kYuvThreadsY);
    count_launch(1);
    if (vector_ok(yuv, L, yuv_frame_stride, cols, bgr, pitch, frame_stride))
        yuv420_to_bgr_kernel<true><<<grid, block, 0, st>>>(yuv, L, yuv_frame_stride, rows, cols, bgr, pitch, frame_stride);
    else
        yuv420_to_bgr_kernel<false><<<grid, block, 0, st>>>(yuv, L, yuv_frame_stride, rows, cols, bgr, pitch, frame_stride);
}

void launch_bgr_to_yuv420(const uint8_t* bgr, size_t pitch, size_t frame_stride, int nframes, int rows, int cols, uint8_t* yuv,
                          const YuvPlanes& L, size_t yuv_frame_stride, cudaStream_t st) {
    if (nframes <= 0) return;
    const dim3 grid = yuv_grid(rows, cols, nframes), block(kYuvThreadsX, kYuvThreadsY);
    count_launch(1);
    if (vector_ok(yuv, L, yuv_frame_stride, cols, bgr, pitch, frame_stride))
        bgr_to_yuv420_kernel<true><<<grid, block, 0, st>>>(bgr, pitch, frame_stride, rows, cols, yuv, L, yuv_frame_stride);
    else
        bgr_to_yuv420_kernel<false><<<grid, block, 0, st>>>(bgr, pitch, frame_stride, rows, cols, yuv, L, yuv_frame_stride);
}

}  // namespace vstabk
