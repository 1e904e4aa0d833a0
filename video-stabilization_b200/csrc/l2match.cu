// K12: exact L2 nearest-neighbour matching of SIFT descriptors on the 5th-generation tensor cores
//   reference: cv::FlannBasedMatcher().match(refDesc, curDesc) + distance filter
//              d <= max(0.5 * mean(d), 0.02)             /root/reference/src/stabilizer.cpp:675-708
// FLANN's randomised KD-trees are approximate and not reproducible call to call (SURVEY A.13); this
// kernel returns the exact nearest neighbour, which equals cv::BFMatcher(NORM_L2).match 100 %:
//   ||a_i - b_j||^2 = ||a_i||^2 + ||b_j||^2 - 2 a_i . b_j
// SIFT descriptors are integers 0..255 (SURVEY A.12): the dot products are exact integers <= 128 * 255^2 = 8.3e6.
//
// l2_nn_i8_kernel: tcgen05 kind::i8 on the raw descriptor bytes (u8 x u8 -> s32), operand tiles by TMA (SWIZZLE_128B: a
// descriptor row is one 128-byte swizzle row), a 4-stage ring of B tiles with full / empty mbarriers, two 128-column TMEM
// accumulators, warp-specialised CTAs (producer lane, MMA lane, four epilogue warps), a whole batch of frames along
// grid.z.  The epilogue folds each 128 x 128 tile into a row-wise arg-min on the packed key (|b|^2 - 2 a.b) * 128 +
// column; the distance matrix never leaves the SM.
#include <cuda.h>
#include "kernels.h"

namespace vstabk {
namespace {

constexpr int TM = 128, TN = 128, TK = 128;          // tile: reference rows, current rows, descriptor length

VSTAB_D unsigned smem_addr(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }

// K-major, SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start address
// >> 4, leading byte offset 0 (one swizzle atom along K), stride byte offset 1024 B (8 rows x 128 B)
// >> 4, version 1 (sm_100), layout type 2 = SWIZZLE_128B.
VSTAB_D unsigned long long umma_desc(unsigned saddr) {
    unsigned long long d = 0;
    d |= (unsigned long long)((saddr >> 4) & 0x3fffu);
    d |= (unsigned long long)((1024u >> 4) & 0x3fffu) << 32;
    d |= 1ull << 46;
    d |= 2ull << 61;
    return d;
}

// ---------------------------------------------------------------------------------------------------------------------
// Pipelined: kind::i8 on the raw descriptor bytes (u8 x u8 -> s32, exact; no conversion pass), operand
// tiles brought in by the TMA engine (cp.async.bulk.tensor.2d, SWIZZLE_128B: a descriptor row IS the 128-byte swizzle
// row), a 4-stage ring of B tiles, two 128-column TMEM accumulators, warp-specialised CTAs of 6 warps:
//   warp 0 (one lane)  TMA producer: A tile once, then B tiles into the ring (full / empty mbarriers)
//   warp 1 (one lane)  MMA issuer: 4 x tcgen05.mma M128 N128 K32 per tile, tcgen05.commit frees the stage and
//                      publishes the accumulator
//   warps 2..5         epilogue: tcgen05.ld of their TMEM lane quarter, min over the tile of the packed key
//                      (|b|^2 - 2 a.b) * 128 + column -- ONE integer multiply-add and one min per element -- then the
//                      tile's winner against the running best (strict <, ascending tiles: lowest index wins ties)
// The grid is (128-row reference tiles) x (splits of the current rows) x (frames), so one frame already fills the
// machine and a batch of frames is one launch; partial results meet in a 64-bit atomicMin on {d2, index}.
constexpr int kStages = 4, kAccs = 2;
constexpr int kTileI8 = TM * 128;                     // 16 KB: 128 rows x 128 bytes
struct __align__(1024) L2Smem {
    unsigned char A[kTileI8];
    unsigned char B[kStages][kTileI8];
    int kc[kAccs][TN];
    unsigned long long full[kStages], empty[kStages], a_full, acc_full[kAccs], acc_empty[kAccs];
    unsigned tmem_base;
};

VSTAB_D void mbar_init(unsigned long long* b, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(b)), "r"(count) : "memory");
}
VSTAB_D void mbar_arrive(unsigned long long* b) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_addr(b)) : "memory");
}
VSTAB_D void mbar_expect_tx(unsigned long long* b, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(b)), "r"(bytes) : "memory");
}
// bounded spin: a protocol error traps (launch failure the host sees) instead of hanging the device
VSTAB_D void mbar_wait(unsigned long long* b, unsigned parity) {
    const unsigned addr = smem_addr(b);
    for (unsigned spin = 0;; ++spin) {
        unsigned done;
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n" : "=r"(done) : "r"(addr), "r"(parity) : "memory");
        if (done) return;
        if (spin > (1u << 26)) __trap();
    }
}
VSTAB_D void tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, unsigned long long* bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(smem_addr(dst)), "l"(map), "r"(smem_addr(bar)), "r"(c0), "r"(c1) : "memory");
}

// per row: squared norm; current rows in [n, round_up(n, 128)) are zeroed (their dot products must be 0: the TMA
// fetches whole tiles), the reference rows' {d2, index} slots are reset
__global__ void __launch_bounds__(256)
l2_prep_kernel(const uint8_t* __restrict__ ref, const int* __restrict__ nref_p, uint8_t* __restrict__ cur, const int* __restrict__ ncur_p,
               int max_kp, size_t cur_frame_stride, int* __restrict__ na, int* __restrict__ nb, unsigned long long* __restrict__ packed) {
    const int frame = blockIdx.y;
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= max_kp) return;
    const int nref = min(nref_p[0], max_kp), ncur = min(ncur_p[frame], max_kp);
    if (row < nref) {
        if (frame == 0) {
            const unsigned w = __ldg(reinterpret_cast<const unsigned*>(ref + (size_t)row * TK) + lane);
            int n = (int)__dp4a(w, w, 0u);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) n += __shfl_xor_sync(0xffffffffu, n, o);
            if (lane == 0) na[row] = n;
        }
        if (lane == 0) packed[(size_t)frame * max_kp + row] = ~0ull;
    }
    uint8_t* crow = cur + (size_t)frame * cur_frame_stride + (size_t)row * TK;
    if (row < ncur) {
        const unsigned w = __ldg(reinterpret_cast<const unsigned*>(crow) + lane);
        int n = (int)__dp4a(w, w, 0u);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) n += __shfl_xor_sync(0xffffffffu, n, o);
        if (lane == 0) nb[(size_t)frame * max_kp + row] = n;
    } else if (row < ((ncur + TN - 1) / TN) * TN) {
        reinterpret_cast<unsigned*>(crow)[lane] = 0u;
    }
}

__global__ void __launch_bounds__(192, 2)
l2_nn_i8_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB,
                const int* __restrict__ nref_p, const int* __restrict__ ncur_p, int max_kp,
                const int* __restrict__ na_g, const int* __restrict__ nb_g, unsigned long long* __restrict__ packed) {
    extern __shared__ unsigned char smem_raw[];
    L2Smem& S = *reinterpret_cast<L2Smem*>(smem_raw + ((1024u - (smem_addr(smem_raw) & 1023u)) & 1023u));
    const int frame = blockIdx.z;
    const int nref = min(nref_p[0], max_kp), ncur = min(ncur_p[frame], max_kp);
    const int row0 = blockIdx.x * TM;
    const int ntiles_all = (ncur + TN - 1) / TN;
    // this CTA's tiles of the current rows: blockIdx.y, blockIdx.y + gridDim.y, ...
    const int ntiles = ntiles_all > (int)blockIdx.y ? (ntiles_all - (int)blockIdx.y + (int)gridDim.y - 1) / (int)gridDim.y : 0;
    if (row0 >= nref || ntiles == 0) return;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < kStages; ++s) { mbar_init(&S.full[s], 1); mbar_init(&S.empty[s], 1); }
#pragma unroll
        for (int a = 0; a < kAccs; ++a) { mbar_init(&S.acc_full[a], 1); mbar_init(&S.acc_empty[a], 4); }
        mbar_init(&S.a_full, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_addr(&S.tmem_base)), "r"(kAccs * TN) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const unsigned tmem = S.tmem_base;

    if (warp == 0) {
        // ================================ TMA producer ================================
        if (lane == 0) {
            mbar_expect_tx(&S.a_full, kTileI8);
            tma_load_2d(S.A, &mapA, 0, row0, &S.a_full);
            for (int it = 0; it < ntiles; ++it) {
                const int s = it % kStages;
                if (it >= kStages) mbar_wait(&S.empty[s], ((it / kStages) - 1) & 1);
                const int j0 = ((int)blockIdx.y + it * (int)gridDim.y) * TN;
                mbar_expect_tx(&S.full[s], kTileI8);
                tma_load_2d(S.B[s], &mapB, 0, frame * max_kp + j0, &S.full[s]);
            }
        }
    } else if (warp == 1) {
        // ================================ MMA issuer ==================================
        if (lane == 0) {
            // instruction descriptor: D = S32 (c_format 2), A = B = unsigned 8-bit (0), both K-major, N, M
            const unsigned idesc = (2u << 4) | ((unsigned)(TN >> 3) << 17) | ((unsigned)(TM >> 4) << 24);
            mbar_wait(&S.a_full, 0);
            for (int it = 0; it < ntiles; ++it) {
                const int s = it % kStages, a = it % kAccs;
                mbar_wait(&S.full[s], (it / kStages) & 1);
                if (it >= kAccs) mbar_wait(&S.acc_empty[a], ((it / kAccs) - 1) & 1);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
                for (int k = 0; k < TK / 32; ++k) {                  // UMMA_K = 32 bytes of 8-bit operands
                    const unsigned long long da = umma_desc(smem_addr(S.A) + k * 32), db = umma_desc(smem_addr(S.B[s]) + k * 32);
                    const unsigned acc = k > 0 ? 1u : 0u;
                    asm volatile(
                        "{\n\t"
                        ".reg .pred p;\n\t"
                        "setp.ne.b32 p, %4, 0;\n\t"
                        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t"
                        "}\n" ::"r"(tmem + (unsigned)(a * TN)), "l"(da), "l"(db), "r"(idesc), "r"(acc) : "memory");
                }
                asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_addr(&S.empty[s])) : "memory");
                asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_addr(&S.acc_full[a])) : "memory");
            }
        }
    } else {
        // ================================ epilogue (warps 2..5) =======================
        const int te = threadIdx.x - 64;                           // 0..127: column this thread prepares
        const int q = warp & 3;                                    // TMEM lane quarter this warp may read
        const int row = row0 + q * 32 + lane;                      // reference row = TMEM lane
        const int na = row < nref ? na_g[row] : 0;
        const int* nbp = nb_g + (size_t)frame * max_kp;
        int bd = 0x7fffffff, bi = -1;
        // |b_j|^2 of this thread's column of the NEXT tile is fetched while the current tile is folded (an L2 round trip
        // in front of the barrier of every tile otherwise: 94 -> 82 us per 64-frame batch)
        auto norm_of = [&](int it) { const int j = ((int)blockIdx.y + it * (int)gridDim.y) * TN + te; return j < ncur ? __ldg(nbp + j) : -1; };
        int nb_next = norm_of(0);
        for (int it = 0; it < ntiles; ++it) {
            const int a = it % kAccs;
            const int j0 = ((int)blockIdx.y + it * (int)gridDim.y) * TN;
            // per-column constant of the packed key: |b_j|^2 * 128 + column (rows beyond the count: zero rows, largest key)
            S.kc[a][te] = nb_next >= 0 ? nb_next * TN + te : 0x7fffffff;
            if (it + 1 < ntiles) nb_next = norm_of(it + 1);
            asm volatile("bar.sync 1, 128;" ::: "memory");
            mbar_wait(&S.acc_full[a], (it / kAccs) & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const unsigned taddr = tmem + (unsigned)(a * TN) + ((unsigned)(q * 32) << 16);
            int bq0 = 0x7fffffff, bq1 = 0x7fffffff, bq2 = 0x7fffffff, bq3 = 0x7fffffff;
            // two register buffers of 32 columns: the TMEM load of the next chunk is in flight while this one is folded
            unsigned r0[32], r1[32];
#define VSTAB_TMEM_LD32(r, col)                                                                                                   \
            asm volatile(                                                                                                         \
                "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "  \
                "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"                         \
                : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),     \
                  "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),          \
                  "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),         \
                  "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])                       \
                : "r"(taddr + (unsigned)(col))                                                                                    \
                : "memory")
#define VSTAB_FOLD32(r, col)                                                                                                      \
            {                                                                                                                     \
                const int4* kc4 = reinterpret_cast<const int4*>(&S.kc[a][col]);                                                   \
                _Pragma("unroll") for (int c = 0; c < 32; c += 4) {                                                               \
                    const int4 k4 = kc4[c >> 2];                                                                                  \
                    bq0 = min(bq0, (int)r[c] * -2 * TN + k4.x);          /* four independent min chains: on a single  */          \
                    bq1 = min(bq1, (int)r[c + 1] * -2 * TN + k4.y);      /* one the fold is bound by its latency      */          \
                    bq2 = min(bq2, (int)r[c + 2] * -2 * TN + k4.z);                                                               \
                    bq3 = min(bq3, (int)r[c + 3] * -2 * TN + k4.w);                                                               \
                }                                                                                                                 \
            }
            VSTAB_TMEM_LD32(r0, 0);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            VSTAB_TMEM_LD32(r1, 32);
            VSTAB_FOLD32(r0, 0)
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            VSTAB_TMEM_LD32(r0, 64);
            VSTAB_FOLD32(r1, 32)
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            VSTAB_TMEM_LD32(r1, 96);
            VSTAB_FOLD32(r0, 64)
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            // the accumulator is in registers: hand it back to the MMA warp before the last fold
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(&S.acc_empty[a]);
            VSTAB_FOLD32(r1, 96)
#undef VSTAB_TMEM_LD32
#undef VSTAB_FOLD32
            const int best = min(min(bq0, bq1), min(bq2, bq3));
            // key = (|b|^2 - 2 a.b) * 128 + column: arithmetic shift recovers the signed value
            const int d2 = na + (best >> 7), j = j0 + (best & (TN - 1));
            if (best != 0x7fffffff && d2 < bd) { bd = d2; bi = j; }
        }
        if (row < nref && bi >= 0)
            atomicMin(&packed[(size_t)frame * max_kp + row], ((unsigned long long)(unsigned)bd << 32) | (unsigned)bi);
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(kAccs * TN) : "memory");
}

// {d2, index} -> the two arrays the filter reads
__global__ void l2_unpack_kernel(const unsigned long long* __restrict__ packed, const int* __restrict__ nref_p, int max_kp,
                                 int* __restrict__ best_idx, int* __restrict__ best_d2) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= min(nref_p[0], max_kp)) return;
    const size_t k = (size_t)blockIdx.y * max_kp + i;                  // blockIdx.y = frame
    const unsigned long long p = packed[k];
    best_idx[k] = p == ~0ull ? -1 : (int)(unsigned)(p & 0xffffffffull);
    best_d2[k] = p == ~0ull ? 0x7fffffff : (int)(unsigned)(p >> 32);
}

// distance filter of the reference (:680-697): d = sqrt(d2) as float (BFMatcher NORM_L2), mean over the
// reference rows in double, keep d <= max(0.5 * mean, 0.02); then gather the point pairs in
// reference order for the similarity fit.  Single CTA.
__global__ void __launch_bounds__(256)
l2_filter_kernel(const int* __restrict__ best_idx, const int* __restrict__ best_d2, const int* __restrict__ nref_p,
                 int nref_max, const int* __restrict__ ncur_p, const OrbKeypoint* __restrict__ ref_kps,
                 const OrbKeypoint* __restrict__ cur_kps, uint8_t* __restrict__ good, float2* __restrict__ ref_pts,
                 float2* __restrict__ cur_pts, uint8_t* __restrict__ status, int* __restrict__ nmatch) {
    __shared__ double wsum_d[8];
    __shared__ int wsum[8];
    __shared__ int s_base;
    __shared__ double s_thr;
    const int nref = min(*nref_p, nref_max);
    const int ncur = *ncur_p;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    double acc = 0.0;
    if (ncur > 0)
        for (int i = threadIdx.x; i < nref; i += 256) acc += (double)__fsqrt_rn((float)best_d2[i]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) wsum_d[wid] = acc;
    if (threadIdx.x == 0) s_base = 0;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int k = 0; k < 8; ++k) t += wsum_d[k];
        const double avg = nref > 0 ? t / (double)nref : 0.0;
        s_thr = fmax(avg * 0.5, 0.02);
    }
    __syncthreads();
    const double thr = s_thr;
    for (int base = 0; base < nref; base += 256) {
        const int i = base + threadIdx.x;
        const bool g = i < nref && ncur > 0 && (double)__fsqrt_rn((float)best_d2[i]) <= thr;
        if (i < nref && good) good[i] = g ? 1 : 0;
        const unsigned ball = __ballot_sync(0xffffffffu, g);
        if (lane == 0) wsum[wid] = __popc(ball);
        __syncthreads();
        int off = s_base;
        for (int k = 0; k < wid; ++k) off += wsum[k];
        if (g && ref_pts) {
            const int pos = off + __popc(ball & ((1u << lane) - 1u));
            const OrbKeypoint a = ref_kps[i], b = cur_kps[best_idx[i]];
            ref_pts[pos] = make_float2(a.x, a.y);
            cur_pts[pos] = make_float2(b.x, b.y);
            status[pos] = 1;
        }
        __syncthreads();
        if (threadIdx.x == 0) { int t = 0; for (int k = 0; k < 8; ++k) t += wsum[k]; s_base += t; }
        __syncthreads();
    }
    if (threadIdx.x == 0 && nmatch) *nmatch = s_base;
}

}  // namespace

// ---- host: tensor maps of the descriptor arrays (u8 [rows][128], SWIZZLE_128B boxes of 128 rows) ---------------------
namespace {
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
bool make_desc_map(CUtensorMap* m, const void* base, size_t rows) {
    static EncodeTiledFn encode = [] {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess) { cudaGetLastError(); fn = nullptr; }
        return (EncodeTiledFn)fn;
    }();
    if (!encode || (reinterpret_cast<uintptr_t>(base) & 15)) return false;
    const cuuint64_t dims[2] = {(cuuint64_t)TK, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)TK};
    const cuuint32_t box[2] = {(cuuint32_t)TK, (cuuint32_t)TN}, estr[2] = {1, 1};
    return encode(m, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
}  // namespace

size_t l2_match_scratch_bytes(int max_kp, int nframes) {
    return (size_t)max_kp * 4 + (size_t)max_kp * nframes * (4 + 8);        // |a|^2, per frame |b|^2 and {d2, index}
}

// `nframes` current sets (cur_desc + f * max_kp * 128, ncur[f]) against ONE reference set: one launch.  Per frame f the
// results land in best_idx / best_d2 + f * max_kp.  false: no tensor map could be made for the descriptor arrays (the
// driver's cuTensorMapEncodeTiled is missing or refused them), nothing was launched.
bool launch_l2_nn_batch(const uint8_t* ref_desc, const int* nref, uint8_t* cur_desc, const int* ncur, int max_kp, int nframes,
                        void* scratch, int* best_idx, int* best_d2, cudaStream_t st) {
    unsigned long long* packed = reinterpret_cast<unsigned long long*>(scratch);
    int* na = reinterpret_cast<int*>(packed + (size_t)max_kp * nframes);
    int* nb = na + max_kp;
    CUtensorMap mapA, mapB;
    if (!make_desc_map(&mapA, ref_desc, (size_t)max_kp) || !make_desc_map(&mapB, cur_desc, (size_t)max_kp * nframes)) return false;
    const int smem = (int)sizeof(L2Smem) + 1024;
    static PerDeviceOnce once;
    once.run([&] { cudaFuncSetAttribute(l2_nn_i8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem); });
    // splits of the current rows: enough CTAs for every SM twice when one frame is matched, fewer per frame in a batch
    const int mt = (max_kp + TM - 1) / TM;
    int splits = (2 * device_sm_count() + mt * nframes - 1) / (mt * nframes);
    splits = splits < 1 ? 1 : (splits > 8 ? 8 : splits);
    count_launch(3);
    l2_prep_kernel<<<dim3((max_kp + 7) / 8, nframes), 256, 0, st>>>(ref_desc, nref, cur_desc, ncur, max_kp, (size_t)max_kp * TK, na, nb, packed);
    l2_nn_i8_kernel<<<dim3(mt, splits, nframes), 192, smem, st>>>(mapA, mapB, nref, ncur, max_kp, na, nb, packed);
    l2_unpack_kernel<<<dim3((max_kp + 255) / 256, nframes), 256, 0, st>>>(packed, nref, max_kp, best_idx, best_d2);
    return true;
}

bool launch_l2_match(const uint8_t* ref_desc, const int* nref, const OrbKeypoint* ref_kps, uint8_t* cur_desc,
                     const int* ncur, const OrbKeypoint* cur_kps, int max_kp, void* scratch, int* best_idx, int* best_d2, uint8_t* good,
                     float2* ref_pts, float2* cur_pts, uint8_t* status, int* nmatch, cudaStream_t st) {
    if (!launch_l2_nn_batch(ref_desc, nref, cur_desc, ncur, max_kp, 1, scratch, best_idx, best_d2, st)) return false;
    count_launch(1);
    l2_filter_kernel<<<1, 256, 0, st>>>(best_idx, best_d2, nref, max_kp, ncur, ref_kps, cur_kps, good, ref_pts, cur_pts, status,
                                        nmatch);
    return true;
}

}  // namespace vstabk
