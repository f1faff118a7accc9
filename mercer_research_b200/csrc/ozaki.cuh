// ozaki.cuh -- f64-grade GEMM on the 5th-generation tensor cores (tcgen05 / TMEM / TMA) by integer slicing.
//
// Why: rcn computes in f64 (rcn/src/rcn.rs:28-31,49) and the parity bar is 1e-9, but tcgen05.mma has no f64 kind, so
// the wide dense layers (BASELINE config 5: 4096-4096-4096, batch 8192; rcn.rs:105-116 forward, :260-314 backprop
// expressed as batched GEMMs, SURVEY.md A.5) would be capped by the 37 TFLOP/s DMMA pipe.  The Ozaki scheme writes
// every operand row as S balanced base-256 digits under a per-row power-of-two scale,
//     x[r,k] = scale[r] * ( q_0[r,k] + sum_{j>=1} d_j[r,k] * 2^(-8j) ),   |q_0| <= 65, d_j in [-128, 127]   (all int8),
// so that every digit-plane product  sum_k a_i[m,k] * b_j[n,k]  is an EXACT int32 dot product on `tcgen05.mma kind::i8`.
// Pairs with equal i+j = d share the weight 2^(-8d) and accumulate into the SAME int32 TMEM accumulator -- still exact
// while 5 * K * 128^2 < 2^31, i.e. K <= 16384 -- and diagonals d > D are dropped: the digits are zero-mean, so what is
// dropped adds up like sqrt(K) and stays ~6e-11 of the result for S = 5, D = 4 (15 int8 MMAs per k-step).
//
// Kernel (one 128 x 96 output tile per CTA, 320 threads, warp-specialised):
//   warp 0      TMA producer: per 64-deep k-block, 5 A-plane boxes (128 x 64 B) + 5 B-plane boxes (96 x 64 B),
//               SWIZZLE_64B, 3-stage ring guarded by full/empty mbarriers;
//   warp 1      TMEM allocator + MMA issuer: one elected thread issues 2 x 15 tcgen05.mma (M128 N96 K32, 8-bit -> s32)
//               per stage into 5 TMEM accumulators (480 of 512 columns), tcgen05.commit frees the smem slot;
//   warps 2-9   epilogue: tcgen05.ld the 5 diagonals, Horner-combine them in f64, apply the row scales and the layer's
//               epilogue functor (bias + sigmoid, sigmoid', store ...), coalesced column-major stores.
// Measured limiter (profiles/): the tensor core's operand fetch from shared memory (SS-mode MMA reads the 128-row A
// tile for every instruction), not L2 or HBM -- hence the widest N tile TMEM allows and the fewest digit planes.
// The planes are produced by ozaki.cu's slicing kernels (HBM-bound: 8 B in, 5 B out per element).
#pragma once
#include <cuda.h>

#include "common.cuh"

namespace rcn {

constexpr int OZ_S = 5;            // digit planes per operand
constexpr int OZ_D = 4;            // highest diagonal kept (i + j <= OZ_D)
constexpr int OZ_BM = 128, OZ_BN = 96, OZ_BK = 64, OZ_STAGES = 3;
constexpr int OZ_MAX_K = 16384;    // exact int32 accumulation bound (see above)
constexpr int OZ_PAIRS = 15;       // digit-plane products per f64 product: |{(i,j): i+j <= OZ_D}|
constexpr int OZ_A_TILE = OZ_BM * OZ_BK;       // bytes of one A slice tile
constexpr int OZ_B_TILE = OZ_BN * OZ_BK;
constexpr int OZ_STAGE_BYTES = OZ_S * (OZ_A_TILE + OZ_B_TILE);
constexpr int OZ_SMEM_BYTES = OZ_STAGES * OZ_STAGE_BYTES + 1024 /* alignment slack */ + 256 /* barriers */;
constexpr int OZ_THREADS = 320;     // warp 0 TMA, warp 1 MMA, warps 2-9 epilogue (two per TMEM lane quadrant)
constexpr int OZ_TMEM_COLS = 512;

struct OzakiWorkspace {
    DevBuf a_slices, b_slices, a_scale, b_scale, partials;
    void release() { a_slices.release(); b_slices.release(); a_scale.release(); b_scale.release(); partials.release(); }
};

// split-K partial store for the tile kernel (split = blockIdx.y): out[split][m*ld_m + n*ld_n]
struct EpiOzSplitStore {
    double* out; size_t ld_m, ld_n, split_stride;
    __device__ __forceinline__ void operator()(int m, int n, double v) const {
        out[(size_t)blockIdx.y * split_stride + (size_t)m * ld_m + (size_t)n * ld_n] = v;
    }
};

// Geometry of an im2col gather (shared with conv.cu): tensor t is [B][Hi][Wi][C] (NHWC); the pixel grid enumerated by the
// GEMM is [B][Ho][Wo]; tap (ky, kx) of grid pixel (oy, ox) reads t[b, oy + ky - ph, ox + kx - pw, :] (zero outside).
struct ConvGeom {
    const double* t;
    int Hi, Wi, C, Ho, Wo, kh, kw, ph, pw;
    int n_pix;   // B * Ho * Wo
    int n_k;     // kh * kw * C
};

// Operand as the GEMM sees it: `rows` x K (rows = M for A, N for B).
//   gather 0: strided matrix; kcontig: element (r, k) at p[r*ld + k], else p[k*ld + r].
//   gather 1 (kcontig): im2col rows -- r = grid pixel (+ pix0), k = (ky, kx, c), c fastest        (conv forward / backward-data)
//   gather 2 (!kcontig): im2col columns -- r = (ky, kx, c), k = grid pixel (+ pix0)             (conv backward-weight)
// Nothing is materialised in f64: the slicing kernels gather straight into the int8 digit planes.
struct OzOperand {
    const double* p;
    size_t ld;
    bool kcontig;
    int gather = 0;
    int pix0 = 0;         // first grid pixel of this (chunk of the) operand
    ConvGeom g{};
};

// A operand gathered by TMA itself (convolution forward / backward-data on NHWC digit planes [S][B][Hi][Wi][C]): the M
// tile is 128 consecutive grid pixels = a (th x tw) patch, k-block kb = (tap, 64-channel block), and the box of tap
// (ky, kx) is the patch shifted by (ky - ph, kx - pw) -- out-of-range rows / columns are zero-filled by the TMA unit,
// which IS the zero padding.  Requires C % 64 == 0 and a pixel grid that tiles into 128-pixel patches.
struct OzConvA {
    int enabled;
    int C, kw, ph, pw, Ho, Wo;
};

// One power-of-two scale per image of a convolution input x [B][per_image] (every pixel of an image, so every im2col row
// the image feeds, shares that image's scale): planes[s][i] for i < B * per_image, scale_out[b] = scale of image b.
// scale_out holds 2 * B doubles (the upper half is scratch for the image maxima).
int ozaki_slice_tensor(const double* x, int B, size_t per_image, int8_t* planes, double* scale_out, cudaStream_t stream);
// 5-D tensor map over planes [OZ_S][B][Hi][Wi][C], box = (64 channels, tw, th, 1, 1), SWIZZLE_64B.
int ozaki_make_conv_tensor_map(CUtensorMap* map, const int8_t* planes, int B, int Hi, int Wi, int C, int tw, int th);

// Slices one operand into int8 planes [OZ_S][rows][Kp] (Kp = K rounded up to 64, zero padded) and scale[rows].
// scale_scratch: `rows` more doubles of scratch (row maxima between the two passes of the row-contiguous variant).
int ozaki_slice(const OzOperand& op, int rows, int K, int Kp, int8_t* planes, double* scale, double* scale_scratch,
                cudaStream_t stream);
// 3-D tensor map over planes [OZ_S][rows][Kp], box = (64 B of k, box_rows, 1 slice), SWIZZLE_64B.
int ozaki_make_tensor_map(CUtensorMap* map, const int8_t* planes, int rows, int Kp, int box_rows);
bool ozaki_available();

// ---- device helpers ------------------------------------------------------------------------------------------------
namespace oz {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t"
        "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void tma_load_5d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3,
                                            int c4) {
    asm volatile(
        "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4) : "memory");
}
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// K-major SWIZZLE_64B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): rows 64 B apart, 8-row groups
// 512 B apart (SBO), LBO = 1 (unused for swizzled K-major), version 1 (Blackwell), layout type 4 (SWIZZLE_64B).
__device__ __forceinline__ uint64_t smem_desc_sw64(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);          // start address, bits [0,14)
    d |= (uint64_t)1 << 16;                              // leading byte offset (16-byte units), bits [16,30)
    d |= (uint64_t)(512 >> 4) << 32;                     // stride byte offset, bits [32,46)
    d |= (uint64_t)1 << 46;                              // descriptor version, bits [46,48)
    d |= (uint64_t)4 << 61;                              // layout type SWIZZLE_64B, bits [61,64)
    return d;
}
// Instruction descriptor (cute::UMMA::InstrDescriptor) for kind::i8: D = s32, A = B = signed int8, both K-major,
// N = 96, M = 128, dense, no saturation.
constexpr uint32_t kInstrDescI8 = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(OZ_BN >> 3) << 17) | ((uint32_t)(OZ_BM >> 4) << 24);

__device__ __forceinline__ void mma_i8(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t"
        "}" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(kInstrDescI8), "r"(accumulate), "r"(0u) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, int32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

}  // namespace oz

// C(m, n) = sum_k A(m, k) B(n, k), delivered to epi(m, n, value).  Tile (blockIdx.x, blockIdx.y) = (m-tile, n-tile).
// (2-CTA clusters that TMA-multicast halves of the A slice into both CTAs were measured neutral -- the kernel is bound by
// shared memory, not by L2 -> SM traffic -- and were removed.)
template <typename Epi>
__global__ void __launch_bounds__(OZ_THREADS, 1) ozaki_gemm_kernel(const __grid_constant__ CUtensorMap map_a,
                                                                    const __grid_constant__ CUtensorMap map_b,
                                                                    const double* __restrict__ scale_a,
                                                                    const double* __restrict__ scale_b, int M, int N, int Kp,
                                                                    int m_tiles, int n_tiles, int kb_per_split,
                                                                    const OzConvA conv, Epi epi) {
    extern __shared__ unsigned char oz_smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(oz_smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + OZ_STAGES * OZ_STAGE_BYTES);
    uint64_t* empty_bar = full_bar + OZ_STAGES;
    uint64_t* tmem_full_bar = empty_bar + OZ_STAGES;
    uint32_t* tmem_base_slot = reinterpret_cast<uint32_t*>(tmem_full_bar + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // rasterisation: groups of 8 m-tiles sweep all n-tiles, so concurrently resident CTAs share operand tiles in L2
    const int tile = blockIdx.x;
    const int group = 8 * n_tiles;
    const int g = tile / group;
    const int g_m0 = g * 8;
    const int g_rows = min(8, m_tiles - g_m0);
    const int in_g = tile - g * group;
    const int m_tile = g_m0 + in_g % g_rows;
    const int n_tile = in_g / g_rows;
    const int m0 = m_tile * OZ_BM, n0 = n_tile * OZ_BN;
    // split-K: blockIdx.y owns k-blocks [kb0, kb0 + n_kb); the epilogue functor sees blockIdx.y and stores a partial
    const int kb0 = blockIdx.y * kb_per_split;
    const int n_kb = min(Kp / OZ_BK - kb0, kb_per_split);

    if (threadIdx.x == 0) {
        for (int s = 0; s < OZ_STAGES; ++s) { oz::mbar_init(full_bar + s, 1); oz::mbar_init(empty_bar + s, 1); }
        oz::mbar_init(tmem_full_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(oz::smem_u32(tmem_base_slot)), "r"(OZ_TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    oz::tc_fence_before();
    __syncthreads();
    oz::tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_base_slot);

    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b) : "memory");
            for (int kb = 0; kb < n_kb; ++kb) {
                const int stage = kb % OZ_STAGES;
                const uint32_t phase = (kb / OZ_STAGES) & 1;
                oz::mbar_wait(empty_bar + stage, phase ^ 1);
                oz::mbar_expect_tx(full_bar + stage, OZ_STAGE_BYTES);
                unsigned char* sa = smem + stage * OZ_STAGE_BYTES;
                unsigned char* sb = sa + OZ_S * OZ_A_TILE;
                if (conv.enabled) {
                    // k-block -> (tap, channel block); tile -> (image, first row, first column) of its pixel patch
                    const int kk = (kb0 + kb) * OZ_BK;
                    const int tap = kk / conv.C, c0 = kk - tap * conv.C;
                    const int ky = tap / conv.kw, kx = tap - ky * conv.kw;
                    const int img = m0 / (conv.Ho * conv.Wo);
                    const int rem = m0 - img * conv.Ho * conv.Wo;
                    const int oy0 = rem / conv.Wo, ox0 = rem - oy0 * conv.Wo;
#pragma unroll
                    for (int s = 0; s < OZ_S; ++s)
                        oz::tma_load_5d(sa + s * OZ_A_TILE, &map_a, full_bar + stage, c0, ox0 + kx - conv.pw, oy0 + ky - conv.ph, img, s);
                } else {
#pragma unroll
                    for (int s = 0; s < OZ_S; ++s) oz::tma_load_3d(sa + s * OZ_A_TILE, &map_a, full_bar + stage, (kb0 + kb) * OZ_BK, m0, s);
                }
#pragma unroll
                for (int s = 0; s < OZ_S; ++s) oz::tma_load_3d(sb + s * OZ_B_TILE, &map_b, full_bar + stage, (kb0 + kb) * OZ_BK, n0, s);
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        if (lane == 0) {
            for (int kb = 0; kb < n_kb; ++kb) {
                const int stage = kb % OZ_STAGES;
                const uint32_t phase = (kb / OZ_STAGES) & 1;
                oz::mbar_wait(full_bar + stage, phase);
                oz::tc_fence_after();
                const uint32_t sa = oz::smem_u32(smem + stage * OZ_STAGE_BYTES);
                const uint32_t sb = sa + OZ_S * OZ_A_TILE;
#pragma unroll
                for (int ks = 0; ks < OZ_BK / 32; ++ks) {
#pragma unroll
                    for (int i = 0; i < OZ_S; ++i) {
                        const uint64_t da = oz::smem_desc_sw64(sa + i * OZ_A_TILE + ks * 32);
#pragma unroll
                        for (int j = 0; j + i <= OZ_D && j < OZ_S; ++j) {
                            const uint64_t db = oz::smem_desc_sw64(sb + j * OZ_B_TILE + ks * 32);
                            // the first MMA into diagonal d = i + j is (kb, ks, i) = (0, 0, 0)
                            oz::mma_i8(tmem_base + (uint32_t)((i + j) * OZ_BN), da, db, (kb | ks | i) != 0 ? 1u : 0u);
                        }
                    }
                }
                oz::tc_commit(empty_bar + stage);   // frees the smem slot once these MMAs have read it
            }
            oz::tc_commit(tmem_full_bar);               // accumulators complete
        }
    } else {
        // ===== epilogue (warps 2..9): TMEM lane quadrant = warp % 4, the two warps of a quadrant split the columns =====
        const int quad = warp & 3;
        const int col_half = (warp - 2) >> 2;
        const int m = m0 + quad * 32 + lane;
        // read while the main loop runs: the slicing kernels that write the scales precede this launch in plain stream
        // order (this kernel is never launched as a programmatic dependent, which would make the read race with them).
        // A TMA-gathered tensor has one scale per image, and a 128-pixel tile never crosses an image (ozaki_conv_tma_ok).
        const double sa = (m < M) ? scale_a[conv.enabled ? m0 / (conv.Ho * conv.Wo) : m] : 0.0;
        oz::mbar_wait(tmem_full_bar, 0);
        oz::tc_fence_after();
        const uint32_t lane_addr = tmem_base + ((uint32_t)(quad * 32) << 16);
        constexpr double kW = 1.0 / 256.0;   // 2^-8 between neighbouring diagonals
#pragma unroll 1
        for (int c0 = col_half * (OZ_BN / 2); c0 < (col_half + 1) * (OZ_BN / 2); c0 += 16) {
            double acc[16];
            {
                int32_t v[16];
                oz::tmem_ld16(lane_addr + (uint32_t)(OZ_D * OZ_BN + c0), v);
                oz::tmem_ld_wait();
#pragma unroll
                for (int q = 0; q < 16; ++q) acc[q] = (double)v[q];
            }
#pragma unroll
            for (int d = OZ_D - 1; d >= 0; --d) {
                int32_t v[16];
                oz::tmem_ld16(lane_addr + (uint32_t)(d * OZ_BN + c0), v);
                oz::tmem_ld_wait();
#pragma unroll
                for (int q = 0; q < 16; ++q) acc[q] = fma(acc[q], kW, (double)v[q]);   // Horner over the diagonals
            }
            if (m < M) {
#pragma unroll
                for (int q = 0; q < 16; ++q) {
                    const int n = n0 + c0 + q;
                    if (n < N) epi(m, n, acc[q] * sa * __ldg(scale_b + n));
                }
            }
        }
        oz::tc_fence_before();
    }
    __syncthreads();
    if (warp == 1) {
        oz::tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(OZ_TMEM_COLS) : "memory");
    }
}

// Host launcher: slices both operands, builds the tensor maps and runs the tile kernel.
// Smallest split count that keeps every split's contraction inside the exact int32 range and, when the output has
// few tiles, spreads the k-blocks over about two waves of CTAs (each split at least 8 k-blocks deep).
inline int ozaki_plan_splits(int M, int N, int K) {
    const int n_kb = (K + OZ_BK - 1) / OZ_BK;
    const long tiles = (long)((M + OZ_BM - 1) / OZ_BM) * ((N + OZ_BN - 1) / OZ_BN);
    int splits = (K + OZ_MAX_K - 1) / OZ_MAX_K;
    if (tiles < kNumSMs) {
        int want = (int)((2L * kNumSMs + tiles - 1) / tiles);
        if (want > n_kb / 8) want = n_kb / 8;
        if (want > splits) splits = want;
    }
    if (splits < 1) splits = 1;
    const int kbps = (n_kb + splits - 1) / splits;
    return (n_kb + kbps - 1) / kbps;
}

// splits > 1: blockIdx.y = split index; `epi` must store a per-split partial (it can read blockIdx.y) that the caller
// then combines in split order.
template <typename Epi>
static int launch_gemm_ozaki(const char* name, const OzOperand& A, const OzOperand& B, int M, int N, int K, const Epi& epi,
                             OzakiWorkspace& ws, cudaStream_t stream, int splits = 1) {
    if (M <= 0 || N <= 0) return RCN_OK;
    const int Kp = ((K + OZ_BK - 1) / OZ_BK) * OZ_BK;
    if (splits < 1) splits = 1;
    const int kb_per_split = (Kp / OZ_BK + splits - 1) / splits;
    splits = (Kp / OZ_BK + kb_per_split - 1) / kb_per_split;
    if (kb_per_split * OZ_BK > OZ_MAX_K)
        return fail(RCN_ERR_INVALID, "tcgen05 integer-slice GEMM: %d k per split exceeds %d (exact int32 accumulation)", kb_per_split * OZ_BK, OZ_MAX_K);
    RCN_TRY(ws.a_slices.reserve((size_t)OZ_S * M * Kp));
    RCN_TRY(ws.b_slices.reserve((size_t)OZ_S * N * Kp));
    RCN_TRY(ws.a_scale.reserve((size_t)2 * M * sizeof(double)));
    RCN_TRY(ws.b_scale.reserve((size_t)2 * N * sizeof(double)));
    RCN_TRY(ozaki_slice(A, M, K, Kp, ws.a_slices.as<int8_t>(), ws.a_scale.as<double>(), ws.a_scale.as<double>() + M, stream));
    RCN_TRY(ozaki_slice(B, N, K, Kp, ws.b_slices.as<int8_t>(), ws.b_scale.as<double>(), ws.b_scale.as<double>() + N, stream));
    const int m_tiles = (M + OZ_BM - 1) / OZ_BM, n_tiles = (N + OZ_BN - 1) / OZ_BN;
    CUtensorMap map_a, map_b;
    RCN_TRY(ozaki_make_tensor_map(&map_a, ws.a_slices.as<int8_t>(), M, Kp, OZ_BM));
    RCN_TRY(ozaki_make_tensor_map(&map_b, ws.b_slices.as<int8_t>(), N, Kp, OZ_BN));
    auto kern = ozaki_gemm_kernel<Epi>;
    static SmemAttrCache attr;
    if (attr.need(OZ_SMEM_BYTES)) RCN_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, OZ_SMEM_BYTES));
    RCN_LAUNCH(name, stream,
               kern<<<dim3((unsigned)(m_tiles * n_tiles), (unsigned)splits), OZ_THREADS, OZ_SMEM_BYTES, stream>>>(
                   map_a, map_b, ws.a_scale.as<double>(), ws.b_scale.as<double>(), M, N, Kp, m_tiles, n_tiles, kb_per_split, OzConvA{}, epi));
    return RCN_OK;
}

// Convolution forward / backward-data with the im2col done by TMA: C(pix, n) = sum_{tap, c} T[pix + tap, c] * Wk(n, (tap, c)).
// `g` describes the gather (ConvGeom); wk is the dense [N][kh*kw*C] weight matrix (k-contiguous).  The tensor is sliced
// ONCE, element-wise (5 B written per element instead of 45 for a materialised im2col), under one scale per image.
// The slicing kernel reads the tensor in 16-byte vectors; a misaligned tensor takes the per-row gather path instead.
inline bool ozaki_conv_tma_ok(const ConvGeom& g) {
    const bool tiles_ok = (g.Wo <= OZ_BM && OZ_BM % g.Wo == 0 && g.Ho % (OZ_BM / g.Wo) == 0) || (g.Wo % OZ_BM == 0);
    return g.C % OZ_BK == 0 && tiles_ok && g.n_k <= OZ_MAX_K && (reinterpret_cast<uintptr_t>(g.t) & 15) == 0;
}

template <typename Epi>
static int launch_conv_ozaki(const char* name, const ConvGeom& g, int B, const double* wk, int N, const Epi& epi, OzakiWorkspace& ws,
                             cudaStream_t stream) {
    const int M = g.n_pix, K = g.n_k;            // K is a multiple of 64 because C is
    if (M <= 0 || N <= 0) return RCN_OK;
    const size_t per_image = (size_t)g.Hi * g.Wi * g.C;
    RCN_TRY(ws.a_slices.reserve((size_t)OZ_S * B * per_image));
    RCN_TRY(ws.b_slices.reserve((size_t)OZ_S * N * K));
    RCN_TRY(ws.a_scale.reserve((size_t)2 * B * sizeof(double)));
    RCN_TRY(ws.b_scale.reserve((size_t)2 * N * sizeof(double)));
    RCN_TRY(ozaki_slice_tensor(g.t, B, per_image, ws.a_slices.as<int8_t>(), ws.a_scale.as<double>(), stream));
    const OzOperand ob{wk, (size_t)K, true};
    RCN_TRY(ozaki_slice(ob, N, K, K, ws.b_slices.as<int8_t>(), ws.b_scale.as<double>(), ws.b_scale.as<double>() + N, stream));
    const int tw = g.Wo < OZ_BM ? g.Wo : OZ_BM, th = OZ_BM / tw;
    CUtensorMap map_a, map_b;
    RCN_TRY(ozaki_make_conv_tensor_map(&map_a, ws.a_slices.as<int8_t>(), B, g.Hi, g.Wi, g.C, tw, th));
    RCN_TRY(ozaki_make_tensor_map(&map_b, ws.b_slices.as<int8_t>(), N, K, OZ_BN));
    auto kern = ozaki_gemm_kernel<Epi>;
    static SmemAttrCache attr;
    if (attr.need(OZ_SMEM_BYTES)) RCN_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, OZ_SMEM_BYTES));
    const int m_tiles = M / OZ_BM, n_tiles = (N + OZ_BN - 1) / OZ_BN;
    const OzConvA conv{1, g.C, g.kw, g.ph, g.pw, g.Ho, g.Wo};
    RCN_LAUNCH(name, stream,
               kern<<<dim3((unsigned)(m_tiles * n_tiles), 1), OZ_THREADS, OZ_SMEM_BYTES, stream>>>(
                   map_a, map_b, ws.a_scale.as<double>(), ws.b_scale.as<double>(), M, N, K, m_tiles, n_tiles, K / OZ_BK, conv, epi));
    return RCN_OK;
}

}  // namespace rcn
