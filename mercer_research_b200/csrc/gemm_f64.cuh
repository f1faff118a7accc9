// gemm_f64.cuh -- the f64 tensor-path GEMM core shared by the dense layers (dense.cu) and the learned-convolution
// extension (conv.cu).
//
//   C(m, n) = sum_k A(m, k) * B(k, n)       k in this split's range, epilogue functor called once per element
//
// tcgen05.mma has no f64 kind, so the f64 tensor path on B200 is the warp-level DMMA (mma.sync.m8n8k4.f64 -> SASS
// DMMA.8x8x4).  Operand tiles are staged through shared memory with cp.async in a 3-stage ring; WHERE an operand
// element comes from is a loader policy: DenseLoader reads a strided matrix, the im2col loaders of conv.cu gather
// NHWC pixels with zero fill, so convolution forward / backward-data / backward-weight run as implicit GEMMs on the
// same main loop without materialising the im2col matrix.
#pragma once
#include "common.cuh"

namespace rcn {

constexpr int KT = 16;       // k depth of one shared-memory tile
constexpr int STAGES = 3;
constexpr int GEMM_THREADS = 256;

template <int ROWS, bool KCONTIG>
struct TileLayout {
    // +4 doubles of pitch: the 4 (k) x 4 (row) doubles a half-warp reads for one DMMA fragment fall into 16
    // distinct 8-byte bank pairs.
    static constexpr int PITCH = KCONTIG ? (KT + 4) : (ROWS + 4);
    static constexpr int ELEMS = KCONTIG ? ROWS * PITCH : KT * PITCH;
    __device__ __forceinline__ static int idx(int r, int kk) { return KCONTIG ? r * PITCH + kk : kk * PITCH + r; }
};

__device__ __forceinline__ void cp_async8(double* smem_dst, const double* gsrc, int src_bytes) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;\n" ::"r"(d), "l"(gsrc), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

// Strided matrix operand.  KCONTIG: element (r, k) at p[r*ld + k]; else at p[k*ld + r].
template <bool KCONTIG_>
struct DenseLoader {
    static constexpr bool KCONTIG = KCONTIG_;
    const double* p;
    int ld;
    int rmax;
    template <int ROWS>
    __device__ __forceinline__ void prepare(int*, int, int) const {}
    template <int ROWS>
    __device__ __forceinline__ void load_tile(double* s, const int*, int r0, int k0, int kmax, int tid) const {
        using TL = TileLayout<ROWS, KCONTIG>;
        constexpr int N = ROWS * KT;
#pragma unroll
        for (int e = tid; e < N; e += GEMM_THREADS) {
            int r, kk;
            if (KCONTIG) { r = e / KT; kk = e % KT; } else { kk = e / ROWS; r = e % ROWS; }
            const bool ok = (r0 + r < rmax) && (k0 + kk < kmax);
            const size_t off = KCONTIG ? (size_t)(r0 + r) * ld + (k0 + kk) : (size_t)(k0 + kk) * ld + (r0 + r);
            cp_async8(s + TL::idx(r, kk), ok ? p + off : p, ok ? 8 : 0);  // src-size 0 => zero fill
        }
    }
    static constexpr int kPrepInts = 0;   // ints of per-CTA row info this loader keeps in shared memory, per row
};

__device__ __forceinline__ void dmma_8x8x4(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

// SLAB: one of several launches over the column tiles, starting at column n_base (unused otherwise, so a grid within the
// gridDim.y limit runs the same code as before slabs existed).
template <int BM, int BN, int WM, int WN, class ALoad, class BLoad, typename Epi, bool SLAB>
__global__ void __launch_bounds__(GEMM_THREADS) gemm_f64_dmma_kernel(const ALoad la, const BLoad lb, int M, int N, int K,
                                                                      int k_per_split, int n_base, Epi epi) {
    static_assert((BM / WM) * (BN / WN) == GEMM_THREADS / 32, "warp grid must use all warps");
    using TA = TileLayout<BM, ALoad::KCONTIG>;
    using TB = TileLayout<BN, BLoad::KCONTIG>;
    constexpr int MF = WM / 8, NF = WN / 8;
    extern __shared__ __align__(16) double smem_gemm[];
    double* sA = smem_gemm;
    double* sB = smem_gemm + STAGES * TA::ELEMS;
    int* infoA = reinterpret_cast<int*>(sB + STAGES * TB::ELEMS);
    int* infoB = infoA + BM * ALoad::kPrepInts;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, t = lane & 3;
    const int wm = warp % (BM / WM), wn = warp / (BM / WM);
    const int m0 = blockIdx.x * BM, n0 = (SLAB ? n_base : 0) + blockIdx.y * BN;
    const int k_begin = blockIdx.z * k_per_split;
    const int k_end = min(K, k_begin + k_per_split);
    const int ntiles = (k_end - k_begin + KT - 1) / KT;

    la.template prepare<BM>(infoA, m0, tid);
    lb.template prepare<BN>(infoB, n0, tid);
    if (ALoad::kPrepInts + BLoad::kPrepInts > 0) __syncthreads();

    double acc[MF][NF][2];
#pragma unroll
    for (int i = 0; i < MF; ++i)
#pragma unroll
        for (int j = 0; j < NF; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

#pragma unroll
    for (int s = 0; s < STAGES - 1; ++s) {
        if (s < ntiles) {
            la.template load_tile<BM>(sA + s * TA::ELEMS, infoA, m0, k_begin + s * KT, k_end, tid);
            lb.template load_tile<BN>(sB + s * TB::ELEMS, infoB, n0, k_begin + s * KT, k_end, tid);
        }
        cp_async_commit();
    }

    for (int kt = 0; kt < ntiles; ++kt) {
        cp_async_wait<STAGES - 2>();
        __syncthreads();  // tile kt landed for everyone; everyone is done reading tile kt-1's slot
        {
            const int nk = kt + STAGES - 1;
            if (nk < ntiles) {
                const int slot = nk % STAGES;
                la.template load_tile<BM>(sA + slot * TA::ELEMS, infoA, m0, k_begin + nk * KT, k_end, tid);
                lb.template load_tile<BN>(sB + slot * TB::ELEMS, infoB, n0, k_begin + nk * KT, k_end, tid);
            }
            cp_async_commit();
        }
        const double* a_s = sA + (kt % STAGES) * TA::ELEMS;
        const double* b_s = sB + (kt % STAGES) * TB::ELEMS;
#pragma unroll
        for (int ks = 0; ks < KT; ks += 4) {
            double af[MF], bf[NF];
#pragma unroll
            for (int i = 0; i < MF; ++i) af[i] = a_s[TA::idx(wm * WM + i * 8 + g, ks + t)];  // A frag: row g, col t
#pragma unroll
            for (int j = 0; j < NF; ++j) bf[j] = b_s[TB::idx(wn * WN + j * 8 + g, ks + t)];  // B frag: row t, col g
#pragma unroll
            for (int i = 0; i < MF; ++i)
#pragma unroll
                for (int j = 0; j < NF; ++j) dmma_8x8x4(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
        }
    }
    cp_async_wait<0>();

    // C frag: row g, cols 2t, 2t+1
#pragma unroll
    for (int i = 0; i < MF; ++i) {
        const int m = m0 + wm * WM + i * 8 + g;
        if (m >= M) continue;
#pragma unroll
        for (int j = 0; j < NF; ++j) {
            const int n = n0 + wn * WN + j * 8 + 2 * t;
            if (n < N) epi(m, n, acc[i][j][0]);
            if (n + 1 < N) epi(m, n + 1, acc[i][j][1]);
        }
    }
}

// Plain one-thread-per-output kernel: slow, obviously correct; cross-checks the DMMA path (RCN_CUDA_GEMM=simt).
// gridDim.y is capped at kMaxGridYZ; the rows of 8 columns beyond it are looped over.
template <bool AK, bool BKc, typename Epi>
__global__ void gemm_f64_simt_kernel(const double* __restrict__ A, int lda, const double* __restrict__ B, int ldb, int M,
                                     int N, int K, int k_per_split, Epi epi) {
    const int m = blockIdx.x * 32 + (threadIdx.x & 31);
    if (m >= M) return;
    const int k_begin = blockIdx.z * k_per_split, k_end = min(K, k_begin + k_per_split);
    for (int n = blockIdx.y * 8 + (threadIdx.x >> 5); n < N; n += gridDim.y * 8) {
        double acc = 0.0;
        for (int k = k_begin; k < k_end; ++k) {
            const double a = AK ? A[(size_t)m * lda + k] : A[(size_t)k * lda + m];
            const double b = BKc ? B[(size_t)n * ldb + k] : B[(size_t)k * ldb + n];
            acc = fma(a, b, acc);
        }
        epi(m, n, acc);
    }
}

template <int BM, int BN, int WM, int WN, class ALoad, class BLoad, typename Epi>
static int launch_dmma(const char* name, const ALoad& la, const BLoad& lb, int M, int N, int K, int splits,
                       int k_per_split, const Epi& epi, cudaStream_t stream) {
    using TA = TileLayout<BM, ALoad::KCONTIG>;
    using TB = TileLayout<BN, BLoad::KCONTIG>;
    constexpr size_t smem = (size_t)STAGES * (TA::ELEMS + TB::ELEMS) * sizeof(double) +
                            (size_t)(BM * ALoad::kPrepInts + BN * BLoad::kPrepInts) * sizeof(int);
    const unsigned n_tiles = cdiv(N, BN);
    if (n_tiles <= kMaxGridYZ) {
        auto kern = gemm_f64_dmma_kernel<BM, BN, WM, WN, ALoad, BLoad, Epi, false>;
        static SmemAttrCache attr;  // per instantiation
        if (attr.need(smem)) RCN_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        const dim3 grid(cdiv(M, BM), n_tiles, splits);
        RCN_LAUNCH(name, stream, kern<<<grid, GEMM_THREADS, smem, stream>>>(la, lb, M, N, K, k_per_split, 0, epi));
        return RCN_OK;
    }
    // More column tiles than gridDim.y holds (a conv layer's columns are its B*Ho*Wo output pixels): one launch per slab
    // of at most kMaxGridYZ tiles.
    auto kern = gemm_f64_dmma_kernel<BM, BN, WM, WN, ALoad, BLoad, Epi, true>;
    static SmemAttrCache attr;
    if (attr.need(smem)) RCN_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    for (unsigned t0 = 0; t0 < n_tiles; t0 += kMaxGridYZ) {
        const dim3 grid(cdiv(M, BM), min(n_tiles - t0, kMaxGridYZ), splits);
        RCN_LAUNCH(name, stream, kern<<<grid, GEMM_THREADS, smem, stream>>>(la, lb, M, N, K, k_per_split, (int)t0 * BN, epi));
    }
    return RCN_OK;
}

// Normalises a split-K request: k_per_split is a multiple of KT, `splits` the number of non-empty splits.
inline void split_plan(int K, int& splits, int& k_per_split) {
    if (splits < 1) splits = 1;
    k_per_split = (K + splits - 1) / splits;
    k_per_split = ((k_per_split + KT - 1) / KT) * KT;
    if (k_per_split < KT) k_per_split = KT;
    splits = K > 0 ? (K + k_per_split - 1) / k_per_split : 1;
}

// Tile-shape dispatch shared by every caller: skinny-M, big, and small-problem tiles.
template <class ALoad, class BLoad, typename Epi>
static int launch_gemm_tiles(const char* name, const ALoad& la, const BLoad& lb, int M, int N, int K, int splits,
                             int k_per_split, const Epi& epi, cudaStream_t stream) {
    if (M <= 32) return launch_dmma<32, 128, 32, 16, ALoad, BLoad, Epi>(name, la, lb, M, N, K, splits, k_per_split, epi, stream);
    const size_t big_tiles = (size_t)cdiv(M, 128) * cdiv(N, 128) * splits;
    if (big_tiles >= (size_t)kNumSMs * 7 / 8)   // (almost) one CTA per SM is enough for the big tile: it is the efficient one
        return launch_dmma<128, 128, 64, 32, ALoad, BLoad, Epi>(name, la, lb, M, N, K, splits, k_per_split, epi, stream);
    return launch_dmma<64, 64, 32, 16, ALoad, BLoad, Epi>(name, la, lb, M, N, K, splits, k_per_split, epi, stream);
}

}  // namespace rcn
