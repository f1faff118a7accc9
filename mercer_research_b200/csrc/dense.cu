// dense.cu -- rcn's fully-connected layers on sm_100a in f64 (the reference computes in f64, so parity is 1e-9).
//
// Reference: rcn/src/rcn.rs:105-116 (forward), :260-314 (backprop), :176-223 (batch sum + SGD), :478-492
// (sigmoid / sigmoid_prime).  The per-sample matvecs / outer products of the reference become three batched
// GEMM shapes (SURVEY.md A.5):
//   forward        A_l     = sigmoid(W_l A_{l-1} + b_l 1^T)
//   backward-data  D_l     = (W_{l+1}^T D_{l+1}) .* s'(Z_l)
//   backward-wt    sum dW_l = D_l A_{l-1}^T ,  sum db_l = D_l 1
// tcgen05.mma has no f64 kind, so the f64 tensor path on B200 is the warp-level DMMA
// (mma.sync.m8n8k4.f64 -> SASS DMMA.8x8x4); operands are staged through shared memory with cp.async in a
// 3-stage ring, accumulators live in registers, bias / sigmoid / sigmoid' / output-delta run in the epilogue.
//
// sigmoid'(z) is evaluated as a*(1-a) with a = sigmoid(z) read back from the stored activation: the reference
// recomputes sigmoid(z) (rcn.rs:491) which is bitwise the same value, and it must NOT be rewritten
// algebraically (1-a cancels for saturated units and parity depends on cancelling identically).
#include "dense.cuh"
#include "gemm_f64.cuh"
#include "opctx.cuh"
#include "ozaki.cuh"

#include <cstdlib>

namespace rcn {

GemmImpl gemm_impl() {
    static int impl = -1;
    if (impl < 0) {
        const char* e = getenv("RCN_CUDA_GEMM");
        impl = !e ? GEMM_AUTO : strcmp(e, "simt") == 0 ? GEMM_SIMT : strcmp(e, "dmma") == 0 ? GEMM_DMMA : strcmp(e, "tc") == 0 ? GEMM_TC : GEMM_AUTO;
    }
    return (GemmImpl)impl;
}

// tcgen05 integer-slice path (ozaki.cuh) when the contraction is really dense: full 128 x 64 tiles, deep K, and enough
// work to amortise slicing both operands; everything else (skinny layers like 4096 -> 10) stays on DMMA.
static bool use_tensor_cores(size_t M, size_t N, size_t K, OzakiWorkspace* oz) {
    if (!oz || !ozaki_available() || K > (size_t)OZ_MAX_K) return false;
    if (gemm_impl() == GEMM_TC) return M >= 1 && N >= 1 && K >= 1;
    if (gemm_impl() != GEMM_AUTO) return false;
    // enough 128 x 96 tiles to occupy at least half of the SMs, and enough work per tile to amortise slicing both operands
    const size_t tiles = ((M + OZ_BM - 1) / OZ_BM) * ((N + OZ_BN - 1) / OZ_BN);
    return M >= 256 && N >= 256 && K >= 512 && tiles >= (size_t)kNumSMs / 2 && (double)M * (double)N * (double)K >= 4.0e9;
}

// rcn.rs:478-483: 1/(1+E^-x).  exp(-x) instead of pow(E,-x): E as an f64 is e*(1-5.3e-17), so the two differ
// by a relative |x|*5.3e-17 -- far inside the 1e-9 parity tolerance.
__device__ __forceinline__ double sigmoid1(double z) { return 1.0 / (1.0 + exp(-z)); }

// ------------------------------------------------------------------------------------------------
// Epilogues.  operator()(m, n, acc) is called once per output element.
// ------------------------------------------------------------------------------------------------
struct EpiForward {
    const double* bias; double* a_out; double* delta_out; const double* onehot; const int64_t* labels; int M;
    __device__ __forceinline__ void operator()(int m, int n, double v) const {
        const double z = v + bias[m];                        // w * a + b           (rcn.rs:287)
        const double a = sigmoid1(z);                        // sigmoid(&z)         (rcn.rs:289)
        const size_t o = (size_t)n * M + m;
        a_out[o] = a;
        if (delta_out) {                                     // (a_L - y) .* sigmoid_prime(z_L)   (rcn.rs:299)
            const double y = onehot ? onehot[o] : ((labels[n] == (int64_t)m) ? 1.0 : 0.0);
            const double sp = a * (1.0 - a);
            delta_out[o] = (a - y) * sp;
        }
    }
};
struct EpiLogits {  // z = w * a + b with no activation: the softmax head's logits (softmax_xent_head_kernel follows)
    const double* bias; double* z_out; int M;
    __device__ __forceinline__ void operator()(int m, int n, double v) const { z_out[(size_t)n * M + m] = v + bias[m]; }
};
struct EpiBackData {
    const double* a; double* delta_out; int M;
    __device__ __forceinline__ void operator()(int m, int n, double v) const {
        const size_t o = (size_t)n * M + m;
        const double s = a[o];
        delta_out[o] = v * (s * (1.0 - s));                  // (W^T delta) .* sigmoid_prime(z)  (rcn.rs:306-308)
    }
};
struct EpiInputGrad {  // dX = W^T delta with no activation derivative: the input gradient of the dense stack
    double* dx; int M;
    __device__ __forceinline__ void operator()(int m, int n, double v) const { dx[(size_t)n * M + m] = v; }
};
struct EpiStore {  // split-K partial (or final) store, column-major M x N
    double* out; int M; size_t split_stride;
    __device__ __forceinline__ void operator()(int m, int n, double v) const {
        out[(size_t)blockIdx.z * split_stride + (size_t)n * M + m] = v;
    }
};

// ------------------------------------------------------------------------------------------------
// Dense GEMM dispatch on the shared DMMA core (gemm_f64.cuh):
//   A(m,k): AK ? A[m*lda + k] : A[k*lda + m]        B(k,n): BKc ? B[n*ldb + k] : B[k*ldb + n]
// ------------------------------------------------------------------------------------------------
template <bool AK, bool BKc, typename Epi>
static int launch_gemm(const char* name, const double* A, int lda, const double* B, int ldb, size_t M_, size_t N_, size_t K_,
                       int splits, const Epi& epi, cudaStream_t stream, OzakiWorkspace* oz = nullptr) {
    if (M_ == 0 || N_ == 0) return RCN_OK;
    if (M_ > 0x7fffffff || N_ > 0x7fffffff || K_ > 0x7fffffff) return fail(RCN_ERR_INVALID, "GEMM dimension too large");
    const int M = (int)M_, N = (int)N_, K = (int)K_;
    if (splits <= 1 && use_tensor_cores(M_, N_, K_, oz)) {
        const OzOperand oa{A, (size_t)lda, AK}, ob{B, (size_t)ldb, BKc};
        return launch_gemm_ozaki(name, oa, ob, M, N, K, epi, *oz, stream);
    }
    int k_per_split;
    split_plan(K, splits, k_per_split);
    if (gemm_impl() == GEMM_SIMT) {
        const dim3 grid(cdiv(M, 32), min(cdiv(N, 8), kMaxGridYZ), splits);
        RCN_LAUNCH(name, stream, gemm_f64_simt_kernel<AK, BKc, Epi><<<grid, 256, 0, stream>>>(A, lda, B, ldb, M, N, K, k_per_split, epi));
        return RCN_OK;
    }
    const DenseLoader<AK> la{A, lda, M};
    const DenseLoader<BKc> lb{B, ldb, N};
    return launch_gemm_tiles(name, la, lb, M, N, K, splits, k_per_split, epi, stream);
}

// Effective split count launch_gemm will use (so callers can size the partial workspace).
static int effective_splits(size_t K, int splits) {
    int k_per_split;
    split_plan((int)K, splits, k_per_split);
    return splits;
}

// ------------------------------------------------------------------------------------------------
// Skinny output layers (rows <= 16, e.g. the 10 classes behind a 4096-wide hidden layer): 20 flop per 8-byte element of
// the wide activation matrix, i.e. HBM-bound streaming work, not a GEMM worth tiling for tensor cores.  Each kernel
// reads the K x N activation matrix exactly once, coalesced, with many independent loads in flight:
//   forward        z = W a + b, sigmoid (+ output delta)     DMMA: a warp owns a K range for 32 samples, W from L2
//   backward-data  delta = (W^T delta_up) .* a (1 - a)       thread = feature, W^T column in registers, 16 samples in flight
//   backward-wt    dW = delta a^T                            thread = feature, 16 accumulators, batch split across CTAs
// ------------------------------------------------------------------------------------------------
constexpr int SK_MAX_ROWS = 16;
constexpr int SK_FWD_SAMPLES = 32;    // samples per CTA of the forward kernel (4 DMMA n-fragments)

__device__ __forceinline__ void sk_dmma(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

// grid = ceil(N / 32); 256 threads: warp w contracts k in [w*K/8, (w+1)*K/8) for the CTA's 32 samples.  A lane loads
// 4 consecutive k of one sample as two 16-byte loads (k = kb + 4t + j, j = 0..3): DMMA k-step j then uses element j of
// every lane, i.e. the k set {kb + 4t + j}, and the W fragment is read at the same k.  Requires K % 128 == 0.
// LOGITS: store z = w * a + b with no activation (the softmax head's logits; delta_out, onehot and labels are unused).
template <bool LOGITS>
__global__ void __launch_bounds__(256) skinny_forward_kernel(const double* __restrict__ W, const double* __restrict__ bias,
                                                             const double* __restrict__ A_in, int M, int K, int N,
                                                             double* __restrict__ A_out, double* __restrict__ delta_out,
                                                             const double* __restrict__ onehot, const int64_t* __restrict__ labels) {
    __shared__ double part[8][SK_FWD_SAMPLES][SK_MAX_ROWS + 1];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, t = lane & 3;
    const int n0 = blockIdx.x * SK_FWD_SAMPLES;
    const int kw = K / 8;
    const int k_lo = warp * kw, k_hi = k_lo + kw;
    double acc[2][4][2];
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
    const double* arow[4];
    bool aok[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int n = n0 + 8 * j + g;
        aok[j] = n < N;
        arow[j] = A_in + (size_t)(aok[j] ? n : 0) * K + 4 * t;
    }
    const bool m0ok = g < M, m1ok = g + 8 < M;
    double2 a[2][4][2];          // two register stages: the loads of block kb + 16 are in flight under the DMMAs of block kb
    double w[2][4][2];
    auto load_block = [&](int st, int kb) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {               // B fragments: 32 bytes per lane and sample
            const double2* p = reinterpret_cast<const double2*>(arow[j] + kb);
            a[st][j][0] = aok[j] ? __ldcs(p) : make_double2(0.0, 0.0);
            a[st][j][1] = aok[j] ? __ldcs(p + 1) : make_double2(0.0, 0.0);
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {               // A fragments: W[m, kb + 4t + q], L2 resident
            const double* wp = W + (size_t)(kb + 4 * t + q) * M + g;
            w[st][q][0] = m0ok ? __ldg(wp) : 0.0;
            w[st][q][1] = m1ok ? __ldg(wp + 8) : 0.0;
        }
    };
    auto mma_block = [&](int st) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            sk_dmma(acc[0][j][0], acc[0][j][1], w[st][0][0], a[st][j][0].x);
            sk_dmma(acc[1][j][0], acc[1][j][1], w[st][0][1], a[st][j][0].x);
            sk_dmma(acc[0][j][0], acc[0][j][1], w[st][1][0], a[st][j][0].y);
            sk_dmma(acc[1][j][0], acc[1][j][1], w[st][1][1], a[st][j][0].y);
            sk_dmma(acc[0][j][0], acc[0][j][1], w[st][2][0], a[st][j][1].x);
            sk_dmma(acc[1][j][0], acc[1][j][1], w[st][2][1], a[st][j][1].x);
            sk_dmma(acc[0][j][0], acc[0][j][1], w[st][3][0], a[st][j][1].y);
            sk_dmma(acc[1][j][0], acc[1][j][1], w[st][3][1], a[st][j][1].y);
        }
    };
    load_block(0, k_lo);
    for (int kb = k_lo; kb < k_hi; kb += 32) {      // K / 8 is a multiple of 16; blocks are taken in pairs (stage 0, stage 1)
        if (kb + 16 < k_hi) load_block(1, kb + 16);
        mma_block(0);
        if (kb + 16 < k_hi) {
            if (kb + 32 < k_hi) load_block(0, kb + 32);
            mma_block(1);
        }
    }
#pragma unroll
    for (int i = 0; i < 2; ++i)                     // C fragment: row g (+8i), samples 8j + 2t, 2t + 1
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            part[warp][8 * j + 2 * t][8 * i + g] = acc[i][j][0];
            part[warp][8 * j + 2 * t + 1][8 * i + g] = acc[i][j][1];
        }
    __syncthreads();
    for (int o = tid; o < SK_FWD_SAMPLES * M; o += 256) {
        const int s = o / M, m = o - s * M;
        const int n = n0 + s;
        if (n >= N) continue;
        double v = part[0][s][m];
#pragma unroll
        for (int q = 1; q < 8; ++q) v += part[q][s][m];          // K ranges in ascending order
        const double z = v + bias[m];                            // w * a + b           (rcn.rs:287)
        if constexpr (LOGITS) {
            A_out[(size_t)n * M + m] = z;
            continue;
        }
        const double act = sigmoid1(z);                          // sigmoid(&z)         (rcn.rs:289)
        const size_t idx = (size_t)n * M + m;
        A_out[idx] = act;
        if (delta_out) {                                         // (a_L - y) .* sigmoid_prime(z_L)   (rcn.rs:299)
            const double y = onehot ? onehot[idx] : ((labels[n] == (int64_t)m) ? 1.0 : 0.0);
            delta_out[idx] = (act - y) * (act * (1.0 - act));
        }
    }
}

// delta_out[k, n] = (sum_m W_up[m, k] delta_up[m, n]) * a (1 - a), a = A[k, n].  grid (ceil(K / 256), chunks of 16
// samples), sample chunks from n_chunk0 on when SLAB (a batch of more chunks than gridDim.y holds is several launches).
template <int MR, bool SLAB>
__global__ void __launch_bounds__(256) skinny_backward_data_kernel(const double* __restrict__ W_up, const double* __restrict__ delta_up,
                                                                   const double* __restrict__ A, int K, int N, int n_chunk0,
                                                                   double* __restrict__ delta_out) {
    constexpr int NS = 16;
    constexpr int MP = (MR + 1) & ~1;               // rows padded to an even count: 16-byte shared loads
    __shared__ __align__(16) double sd[NS][MP];
    const int k = blockIdx.x * 256 + threadIdx.x;
    const int n0 = ((SLAB ? n_chunk0 : 0) + blockIdx.y) * NS;
    for (int i = threadIdx.x; i < NS * MP; i += 256) {
        const int s = i / MP, m = i - s * MP;
        sd[s][m] = (m < MR && n0 + s < N) ? delta_up[(size_t)(n0 + s) * MR + m] : 0.0;
    }
    double w[MR];
    if (k < K) {
#pragma unroll
        for (int m = 0; m < MR; ++m) w[m] = __ldg(W_up + (size_t)k * MR + m);
    }
    __syncthreads();
    if (k >= K) return;
    double a[NS];
#pragma unroll
    for (int s = 0; s < NS; ++s) a[s] = (n0 + s < N) ? __ldcs(A + (size_t)(n0 + s) * K + k) : 0.0;
#pragma unroll
    for (int s = 0; s < NS; ++s) {
        if (n0 + s < N) {
            double v = 0.0;
#pragma unroll
            for (int m = 0; m < MR; m += 2) {                               // W^T delta, m ascending
                const double2 dd = *reinterpret_cast<const double2*>(&sd[s][m]);
                v = fma(w[m], dd.x, v);
                if (m + 1 < MR) v = fma(w[m + 1], dd.y, v);
            }
            __stcs(delta_out + (size_t)(n0 + s) * K + k, v * (a[s] * (1.0 - a[s])));   // .* sigmoid_prime(z)  (rcn.rs:306-308)
        }
    }
}

// partial[split][m + k*MR] = sum over this split's samples of delta[m, n] * A_prev[k, n].  grid (ceil(K / 256), splits).
template <int MR>
__global__ void __launch_bounds__(256) skinny_backward_weight_kernel(const double* __restrict__ delta, const double* __restrict__ A_prev,
                                                                     int K, int N, int n_per_split, double* __restrict__ partial) {
    constexpr int NS = 16;
    constexpr int MP = (MR + 1) & ~1;
    __shared__ __align__(16) double sd[2][NS][MP];
    const int k = blockIdx.x * 256 + threadIdx.x;
    const int n_lo = blockIdx.y * n_per_split, n_hi = min(N, n_lo + n_per_split);
    const bool kok = k < K;
    double acc[MR];
#pragma unroll
    for (int m = 0; m < MR; ++m) acc[m] = 0.0;
    // (a two-stage register pipeline over the chunks was measured slower here: 126 registers, 83.7 vs 75.7 us on c5)
    int buf = 0;
    for (int nb = n_lo; nb < n_hi; nb += NS, buf ^= 1) {
        for (int i = threadIdx.x; i < NS * MP; i += 256) {
            const int s = i / MP, m = i - s * MP;
            sd[buf][s][m] = (m < MR && nb + s < n_hi) ? delta[(size_t)(nb + s) * MR + m] : 0.0;
        }
        double a[NS];
#pragma unroll
        for (int s = 0; s < NS; ++s) a[s] = (kok && nb + s < n_hi) ? __ldcs(A_prev + (size_t)(nb + s) * K + k) : 0.0;
        __syncthreads();   // this chunk's deltas are staged; the other buffer is free again
#pragma unroll
        for (int s = 0; s < NS; ++s)
#pragma unroll
            for (int m = 0; m < MR; m += 2) {                                         // samples in ascending order
                const double2 dd = *reinterpret_cast<const double2*>(&sd[buf][s][m]);
                acc[m] = fma(dd.x, a[s], acc[m]);
                if (m + 1 < MR) acc[m + 1] = fma(dd.y, a[s], acc[m + 1]);
            }
    }
    if (kok) {
        double* out = partial + (size_t)blockIdx.y * K * MR + (size_t)k * MR;
#pragma unroll
        for (int m = 0; m < MR; ++m) out[m] = acc[m];
    }
}

static bool skinny_layer(size_t M, size_t K) {
    return gemm_impl() == GEMM_AUTO && M >= 1 && M <= (size_t)SK_MAX_ROWS && K >= 512 && K % 128 == 0;
}

template <int MR>
static int launch_skinny_bwd_t(const double* W_up, const double* delta_up, const double* A, size_t M, size_t K, size_t N,
                               double* delta_out, cudaStream_t stream) {
    const unsigned chunks = cdiv(N, 16);
    if (chunks <= kMaxGridYZ) {
        RCN_LAUNCH("skinny_backward_data_kernel", stream,
                   skinny_backward_data_kernel<MR, false><<<dim3(cdiv(M, 256), chunks), 256, 0, stream>>>(W_up, delta_up, A, (int)M,
                                                                                                      (int)N, 0, delta_out));
        return RCN_OK;
    }
    for (unsigned c0 = 0; c0 < chunks; c0 += kMaxGridYZ)   // one launch per slab of at most kMaxGridYZ sample chunks
        RCN_LAUNCH("skinny_backward_data_kernel", stream,
                   skinny_backward_data_kernel<MR, true><<<dim3(cdiv(M, 256), min(chunks - c0, kMaxGridYZ)), 256, 0, stream>>>(
                       W_up, delta_up, A, (int)M, (int)N, (int)c0, delta_out));
    return RCN_OK;
}

// ------------------------------------------------------------------------------------------------
// Layer entry points
// ------------------------------------------------------------------------------------------------
int launch_dense_forward(const double* W, const double* b, const double* A_in, size_t M, size_t K, size_t N,
                         double* A_out, double* delta_out, const double* onehot, const int64_t* labels,
                         cudaStream_t stream, OzakiWorkspace* oz) {
    // the skinny kernel reads A_in as double2: a layer's activations start at an odd double when the rows below it times B
    // are odd, and those take the GEMM, whose cp.async copies are 8 bytes
    if (N > 0 && skinny_layer(M, K) && ((uintptr_t)A_in & 15) == 0) {
        RCN_LAUNCH("skinny_forward_kernel", stream,
                   skinny_forward_kernel<false><<<cdiv(N, SK_FWD_SAMPLES), 256, 0, stream>>>(W, b, A_in, (int)M, (int)K, (int)N, A_out,
                                                                                             delta_out, onehot, labels));
        return RCN_OK;
    }
    EpiForward epi{b, A_out, delta_out, onehot, labels, (int)M};
    const bool tc = use_tensor_cores(M, N, K, oz);
    return launch_gemm<false, true, EpiForward>(tc ? "dense_forward_gemm(tcgen05 int8 slices)" : "dense_forward_gemm", W, (int)M, A_in,
                                                (int)K, M, N, K, 1, epi, stream, oz);
}

int launch_dense_logits(const double* W, const double* b, const double* A_in, size_t M, size_t K, size_t N, double* Z,
                        cudaStream_t stream, OzakiWorkspace* oz) {
    if (N > 0 && skinny_layer(M, K) && ((uintptr_t)A_in & 15) == 0) {   // 16-byte loads, as in launch_dense_forward
        RCN_LAUNCH("skinny_forward_kernel(logits)", stream,
                   skinny_forward_kernel<true><<<cdiv(N, SK_FWD_SAMPLES), 256, 0, stream>>>(W, b, A_in, (int)M, (int)K, (int)N, Z,
                                                                                            nullptr, nullptr, nullptr));
        return RCN_OK;
    }
    EpiLogits epi{b, Z, (int)M};
    const bool tc = use_tensor_cores(M, N, K, oz);
    return launch_gemm<false, true, EpiLogits>(tc ? "dense_logits_gemm(tcgen05 int8 slices)" : "dense_logits_gemm", W, (int)M, A_in,
                                               (int)K, M, N, K, 1, epi, stream, oz);
}

int launch_dense_backward_data(const double* W_up, const double* delta_up, const double* A, size_t M, size_t K,
                               size_t N, double* delta_out, cudaStream_t stream, OzakiWorkspace* oz) {
    // here M = width of the layer below (features), K = rows of the upper layer (the contraction)
    if (N > 0 && M > 0 && skinny_layer(K, M)) {
        switch (K) {
#define RCN_SK_CASE(R) case R: return launch_skinny_bwd_t<R>(W_up, delta_up, A, M, K, N, delta_out, stream);
            RCN_SK_CASE(1) RCN_SK_CASE(2) RCN_SK_CASE(3) RCN_SK_CASE(4) RCN_SK_CASE(5) RCN_SK_CASE(6) RCN_SK_CASE(7) RCN_SK_CASE(8)
            RCN_SK_CASE(9) RCN_SK_CASE(10) RCN_SK_CASE(11) RCN_SK_CASE(12) RCN_SK_CASE(13) RCN_SK_CASE(14) RCN_SK_CASE(15) RCN_SK_CASE(16)
#undef RCN_SK_CASE
            default: break;
        }
    }
    EpiBackData epi{A, delta_out, (int)M};
    // A(m,k) = W_up[k, m]; W_up is K x M column-major => k-contiguous with lda = K.
    const bool tc = use_tensor_cores(M, N, K, oz);
    return launch_gemm<true, true, EpiBackData>(tc ? "dense_backward_data_gemm(tcgen05 int8 slices)" : "dense_backward_data_gemm", W_up,
                                                (int)K, delta_up, (int)K, M, N, K, 1, epi, stream, oz);
}

int launch_dense_input_grad(const double* W0, const double* delta0, size_t M, size_t K, size_t N, double* dx, cudaStream_t stream,
                            OzakiWorkspace* oz) {
    EpiInputGrad epi{dx, (int)M};
    const bool tc = use_tensor_cores(M, N, K, oz);   // the engine choice of launch_dense_backward_data
    return launch_gemm<true, true, EpiInputGrad>(tc ? "dense_input_grad_gemm(tcgen05 int8 slices)" : "dense_input_grad_gemm", W0,
                                                 (int)K, delta0, (int)K, M, N, K, 1, epi, stream, oz);
}

__global__ void reduce_splits_kernel(const double* __restrict__ part, int splits, size_t n, double* __restrict__ out) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        double s = 0.0;
        for (int p0 = 0; p0 < splits; p0 += 8) {          // 8 loads in flight, added in split order (deterministic)
            double v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) v[u] = (p0 + u < splits) ? __ldcs(part + (size_t)(p0 + u) * n + i) : 0.0;
#pragma unroll
            for (int u = 0; u < 8; ++u) if (p0 + u < splits) s = (p0 + u == 0) ? v[u] : s + v[u];
        }
        out[i] = s;
    }
}

// db[m] = sum_n delta[m, n].  Grid (row blocks of 32, column splits): lane = row, warp = column phase inside the CTA's
// column range, 4 loads in flight per thread; per-CTA partials meet in the scratch buffer and the last CTA of a row
// block to arrive adds them in split order (deterministic, no atomics on the data).
__global__ void __launch_bounds__(256) bias_grad_kernel(const double* __restrict__ delta, int M, int N, int n_per_split,
                                                        double* __restrict__ db, double* __restrict__ partial,
                                                        unsigned* __restrict__ tickets) {
    __shared__ double sm[8][33];
    __shared__ bool s_last;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int m = blockIdx.x * 32 + lane;
    const int S = gridDim.y;
    const int n_lo = blockIdx.y * n_per_split, n_hi = min(N, n_lo + n_per_split);
    double acc = 0.0;
    if (m < M) {
        for (int n = n_lo + w; n < n_hi; n += 128) {
            double v[16];
#pragma unroll
            for (int u = 0; u < 16; ++u) v[u] = (n + 8 * u < n_hi) ? __ldcs(delta + (size_t)(n + 8 * u) * M + m) : 0.0;
#pragma unroll
            for (int u = 0; u < 16; ++u) acc += v[u];
        }
    }
    sm[w][lane] = acc;
    __syncthreads();
    if (w == 0) {
        double s = sm[0][lane];
#pragma unroll
        for (int i = 1; i < 8; ++i) s += sm[i][lane];
        if (S == 1) { if (m < M) db[m] = s; return; }
        if (m < M) partial[(size_t)blockIdx.y * M + m] = s;
    }
    if (S == 1) return;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned t = atomicAdd(tickets + blockIdx.x, 1u);
        s_last = (t == (unsigned)S - 1);
        if (s_last) tickets[blockIdx.x] = 0;
    }
    __syncthreads();
    if (s_last && w == 0 && m < M) {
        __threadfence();
        double s = 0.0;
        for (int q0 = 0; q0 < S; q0 += 8) {               // 8 loads in flight, added in split order (deterministic)
            double v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) v[u] = (q0 + u < S) ? __ldcg(partial + (size_t)(q0 + u) * M + m) : 0.0;
#pragma unroll
            for (int u = 0; u < 8; ++u) if (q0 + u < S) s += v[u];
        }
        db[m] = s;
    }
}

// Wide layers (M >= 256): thread = row, a CTA owns 256 consecutive rows (2 KB contiguous per column: whole DRAM bursts
// instead of 256-byte islands 8 * M bytes apart) and a column range, 16 loads in flight per thread; per-CTA partials are
// added in split order by the last CTA of the row block to arrive (deterministic).
__global__ void __launch_bounds__(256) bias_grad_wide_kernel(const double* __restrict__ delta, int M, int N, int n_per_split,
                                                             double* __restrict__ db, double* __restrict__ partial,
                                                             unsigned* __restrict__ tickets) {
    __shared__ bool s_last;
    const int m = blockIdx.x * 256 + threadIdx.x;
    const int S = gridDim.y;
    const int n_lo = blockIdx.y * n_per_split, n_hi = min(N, n_lo + n_per_split);
    double acc = 0.0;
    if (m < M) {
        for (int n = n_lo; n < n_hi; n += 16) {
            double v[16];
#pragma unroll
            for (int u = 0; u < 16; ++u) v[u] = (n + u < n_hi) ? __ldcs(delta + (size_t)(n + u) * M + m) : 0.0;
#pragma unroll
            for (int u = 0; u < 16; ++u) acc += v[u];
        }
        if (S == 1) db[m] = acc; else partial[(size_t)blockIdx.y * M + m] = acc;
    }
    if (S == 1) return;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned t = atomicAdd(tickets + blockIdx.x, 1u);
        s_last = (t == (unsigned)S - 1);
        if (s_last) tickets[blockIdx.x] = 0;
    }
    __syncthreads();
    if (s_last && m < M) {
        __threadfence();
        double s = 0.0;
        for (int q0 = 0; q0 < S; q0 += 8) {               // 8 loads in flight, added in split order (deterministic)
            double v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) v[u] = (q0 + u < S) ? __ldcg(partial + (size_t)(q0 + u) * M + m) : 0.0;
#pragma unroll
            for (int u = 0; u < 8; ++u) if (q0 + u < S) s += v[u];
        }
        db[m] = s;
    }
}

int launch_reduce_splits(const double* partials, int splits, size_t n, double* out, cudaStream_t stream) {
    unsigned grid = cdiv(n, 256);
    if (grid > kNumSMs * 8) grid = kNumSMs * 8;
    RCN_LAUNCH("reduce_splits_kernel", stream, reduce_splits_kernel<<<grid, 256, 0, stream>>>(partials, splits, n, out));
    return RCN_OK;
}

int launch_bias_grad(const double* delta, size_t M, size_t N, double* db, ReduceScratch& rs, cudaStream_t stream) {
    if (M == 0) return RCN_OK;
    if (M >= 256 && cdiv(M, 256) <= 1023) {
        const unsigned rb = cdiv(M, 256);
        unsigned S = (4 * kNumSMs + rb - 1) / rb;
        const unsigned max_s = (unsigned)((N + 63) / 64);
        if (S > max_s) S = max_s;
        if (S < 1) S = 1;
        int n_per_split = (int)((N + S - 1) / S);
        n_per_split = (n_per_split + 15) / 16 * 16;
        S = (unsigned)((N + n_per_split - 1) / n_per_split);
        if (S < 1) S = 1;
        RCN_TRY(rs.ensure((size_t)S * M * sizeof(double), stream));
        RCN_LAUNCH("bias_grad_kernel", stream,
                   bias_grad_wide_kernel<<<dim3(rb, S), 256, 0, stream>>>(delta, (int)M, (int)N, n_per_split, db, rs.partials(), rs.tickets()));
        return RCN_OK;
    }
    const unsigned row_blocks = cdiv(M, 32);
    if (row_blocks > 1023) return fail(RCN_ERR_INVALID, "layer too wide for the bias-gradient reduction");
    // enough column splits to cover the machine a few times over, each at least 256 columns deep
    unsigned S = (4 * kNumSMs + row_blocks - 1) / row_blocks;
    const unsigned max_s = (unsigned)((N + 255) / 256);
    if (S > max_s) S = max_s;
    if (S < 1) S = 1;
    int n_per_split = (int)((N + S - 1) / S);
    n_per_split = (n_per_split + 31) / 32 * 32;
    S = (unsigned)((N + n_per_split - 1) / n_per_split);
    if (S < 1) S = 1;
    RCN_TRY(rs.ensure((size_t)S * M * sizeof(double), stream));
    RCN_LAUNCH("bias_grad_kernel", stream,
               bias_grad_kernel<<<dim3(row_blocks, S), 256, 0, stream>>>(delta, (int)M, (int)N, n_per_split, db, rs.partials(), rs.tickets()));
    return RCN_OK;
}

int launch_dense_backward_weight(const double* delta, const double* A_prev, size_t M, size_t N, size_t Kb, double* dW,
                                 double* db, DevBuf& workspace, ReduceScratch& rs, cudaStream_t stream, OzakiWorkspace* oz) {
    if (M == 0) return RCN_OK;
    if (N > 0 && Kb > 0 && skinny_layer(M, N)) {
        // thread = input feature, batch split across CTAs; the partials are added in split order (deterministic)
        int splits = (int)((4 * (size_t)kNumSMs + cdiv(N, 256) - 1) / cdiv(N, 256));
        const int max_splits = (int)((Kb + 63) / 64);
        if (splits > max_splits) splits = max_splits;
        if (splits < 1) splits = 1;
        int n_per_split = (int)((Kb + splits - 1) / splits);
        n_per_split = (n_per_split + 15) / 16 * 16;
        splits = (int)((Kb + n_per_split - 1) / n_per_split);
        RCN_TRY(workspace.reserve((size_t)splits * M * N * sizeof(double)));
        double* part = workspace.as<double>();
        const dim3 grid(cdiv(N, 256), splits);
        switch (M) {
#define RCN_SK_CASE(R) case R: RCN_LAUNCH("skinny_backward_weight_kernel", stream, skinny_backward_weight_kernel<R><<<grid, 256, 0, stream>>>(delta, A_prev, (int)N, (int)Kb, n_per_split, part)); break;
            RCN_SK_CASE(1) RCN_SK_CASE(2) RCN_SK_CASE(3) RCN_SK_CASE(4) RCN_SK_CASE(5) RCN_SK_CASE(6) RCN_SK_CASE(7) RCN_SK_CASE(8)
            RCN_SK_CASE(9) RCN_SK_CASE(10) RCN_SK_CASE(11) RCN_SK_CASE(12) RCN_SK_CASE(13) RCN_SK_CASE(14) RCN_SK_CASE(15) RCN_SK_CASE(16)
#undef RCN_SK_CASE
            default: return fail(RCN_ERR_INVALID, "internal: skinny layer with %zu rows", M);
        }
        RCN_TRY(launch_reduce_splits(part, splits, M * N, dW, stream));
        return launch_bias_grad(delta, M, Kb, db, rs, stream);
    }
    if (N > 0 && use_tensor_cores(M, N, Kb, oz)) {
        // enough output tiles to fill the machine without splitting the batch: one exact pass, deterministic by construction
        EpiStore epi{dW, (int)M, 0};
        RCN_TRY((launch_gemm<false, false, EpiStore>("dense_backward_weight_gemm(tcgen05 int8 slices)", delta, (int)M, A_prev, (int)N, M,
                                                     N, Kb, 1, epi, stream, oz)));
        return launch_bias_grad(delta, M, Kb, db, rs, stream);
    }
    // Split the batch (K) dimension so the small M x N output still fills the machine; partials are summed in
    // a fixed order (deterministic, unlike the reference's mutex-ordered sum, rcn.rs:190-205).
    size_t tiles;
    if (M <= 32) tiles = (size_t)cdiv(M, 32) * cdiv(N, 128);
    else {
        tiles = (size_t)cdiv(M, 128) * cdiv(N, 128);
        if (tiles < (size_t)kNumSMs) tiles = (size_t)cdiv(M, 64) * cdiv(N, 64);
    }
    int splits = 1;
    if (tiles < (size_t)kNumSMs && N > 0) {
        splits = (int)((2 * kNumSMs + tiles - 1) / tiles);
        const int max_splits = (int)(Kb / 64) > 0 ? (int)(Kb / 64) : 1;
        if (splits > max_splits) splits = max_splits;
        if (splits > 64) splits = 64;
        // Few 128 x 128 tiles but a deep batch (c3: dW0 is 256 x 1024 over 4096 samples = 16 tiles): ONE wave of the big tile
        // -- one CTA per SM, 32 DMMAs per 12 fragment loads; 0.86 of the DGEMM peak at one CTA per SM on the c5 shapes --
        // with the batch split floor(148 / tiles) ways beats two waves of 64 x 64 tiles (ncu, c3: 20 % warps active, 0.52 of peak).
        // launch_gemm_tiles takes the big tile when tiles x splits covers at least 7/8 of the SMs.
        const size_t big = M > 32 ? (size_t)cdiv(M, 128) * cdiv(N, 128) : 0;
        if (big > 0 && big < (size_t)kNumSMs) {
            const int s_big = (int)((size_t)kNumSMs / big);
            if (s_big >= 2 && Kb / (size_t)s_big >= 256 && big * (size_t)s_big >= (size_t)kNumSMs * 7 / 8) splits = s_big;
        }
    }
    splits = effective_splits(Kb, splits);
    if (N > 0) {
        if (splits == 1) {
            EpiStore epi{dW, (int)M, 0};
            RCN_TRY((launch_gemm<false, false, EpiStore>("dense_backward_weight_gemm", delta, (int)M, A_prev, (int)N, M, N, Kb, 1, epi, stream)));
        } else {
            RCN_TRY(workspace.reserve((size_t)splits * M * N * sizeof(double)));
            EpiStore epi{workspace.as<double>(), (int)M, M * N};
            RCN_TRY((launch_gemm<false, false, EpiStore>("dense_backward_weight_gemm", delta, (int)M, A_prev, (int)N, M, N, Kb, splits, epi, stream)));
            RCN_TRY(launch_reduce_splits(workspace.as<double>(), splits, M * N, dW, stream));
        }
    }
    return launch_bias_grad(delta, M, Kb, db, rs, stream);
}

// ------------------------------------------------------------------------------------------------
// SGD step, argmax, batch statistics
// ------------------------------------------------------------------------------------------------
__global__ void sgd_update_kernel(double* __restrict__ p, const double* __restrict__ g, size_t n, double scale,
                                  long long* __restrict__ cursor, long long batch, long long n_samples,
                                  const double* __restrict__ stats, double* __restrict__ stats_ring) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        p[i] = sgd_apply(p[i], scale, g[i]);  // &lw.0 - (eta / B) * w   (rcn.rs:214,221): product rounded, then subtracted
    if (cursor && blockIdx.x == 0 && threadIdx.x == 0) {
        if (stats_ring) {   // this step's {cost, hits} straight into the (pinned host) result ring: one 16-byte write
            double* dst = stats_ring + 2 * (*cursor / batch);
            dst[0] = stats[0];
            dst[1] = stats[1];
        }
        // next chunk of training_set.chunks_exact(batch) (rcn.rs:147); the remainder is dropped, then wrap
        long long c = *cursor + batch;
        if (c + batch > n_samples) c = 0;
        *cursor = c;
    }
}

int launch_sgd_update(double* params, const double* grads, size_t n, double scale, cudaStream_t stream,
                      long long* cursor, long long batch, long long n_samples, const double* stats, double* stats_ring) {
    if (n == 0 && !cursor) return RCN_OK;
    unsigned grid = n ? cdiv(n, 256) : 1;   // n == 0 with a cursor: only the cursor advances
    if (grid > kNumSMs * 8) grid = kNumSMs * 8;
    RCN_LAUNCH("sgd_update_kernel", stream,
               sgd_update_kernel<<<grid, 256, 0, stream>>>(params, grads, n, scale, cursor, batch, n_samples, stats, stats_ring));
    return RCN_OK;
}

__global__ void argmax_last_kernel(const double* __restrict__ acts, int n, size_t B, int64_t* __restrict__ labels) {
    for (size_t b = blockIdx.x * (size_t)blockDim.x + threadIdx.x; b < B; b += (size_t)gridDim.x * blockDim.x) {
        const double* a = acts + b * n;
        int best = 0;
        double bv = a[0];
        for (int i = 1; i < n; ++i) {
            const double v = a[i];
            if (!(v < bv)) { bv = v; best = i; }  // max_by(total_cmp): last maximal element wins (rcn.rs:92-97)
        }
        labels[b] = best;
    }
}

int launch_argmax_last(const double* acts, size_t n, size_t B, int64_t* labels, cudaStream_t stream) {
    if (B == 0) return RCN_OK;
    unsigned grid = cdiv(B, 128);
    if (grid > kNumSMs * 8) grid = kNumSMs * 8;
    RCN_LAUNCH("argmax_last_kernel", stream, argmax_last_kernel<<<grid, 128, 0, stream>>>(acts, (int)n, B, labels));
    return RCN_OK;
}

// cost = sum_b 0.5*|a-y|^2; hits per rcn.rs:153-157: the set {i : a_i == max a} must equal {label}.  One thread per
// sample, 256 samples per CTA; per-CTA partials are added in CTA order by the last CTA to arrive => deterministic.
__global__ void __launch_bounds__(256) batch_stats_kernel(const double* __restrict__ acts, int n, size_t B,
                                                         const double* __restrict__ onehot,
                                                         const int64_t* __restrict__ labels, double* __restrict__ stats,
                                                         double* __restrict__ partial, unsigned* __restrict__ ticket) {
    __shared__ double sc[256];
    __shared__ unsigned long long sh[256];
    __shared__ bool s_last;
    double cost = 0.0;
    unsigned long long hits = 0;
    const size_t b = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    if (b < B) {
        const double* a = acts + b * n;
        double mx = a[0];
        for (int i = 1; i < n; ++i) mx = fmax(mx, a[i]);
        bool ok = true;
        double c = 0.0;
        for (int i = 0; i < n; ++i) {
            const double y = onehot ? onehot[b * n + i] : ((labels[b] == (int64_t)i) ? 1.0 : 0.0);
            const double d = a[i] - y;
            c += d * d;
            const double r = (a[i] == mx) ? 1.0 : 0.0;
            ok = ok && (r == y);
        }
        cost = 0.5 * c;
        hits = ok ? 1ull : 0ull;
    }
    sc[threadIdx.x] = cost;
    sh[threadIdx.x] = hits;
    __syncthreads();
    if (threadIdx.x == 0) {
        double ct = 0.0;
        unsigned long long ht = 0;
        for (int i = 0; i < 256; ++i) { ct += sc[i]; ht += sh[i]; }
        partial[2 * blockIdx.x] = ct;
        reinterpret_cast<unsigned long long*>(partial)[2 * blockIdx.x + 1] = ht;
        __threadfence();
        const unsigned t = atomicAdd(ticket, 1u);
        s_last = (t == gridDim.x - 1);
        if (s_last) *ticket = 0;
    }
    __syncthreads();
    if (s_last && threadIdx.x == 0) {
        __threadfence();
        double ct = 0.0;
        unsigned long long ht = 0;
        for (unsigned i = 0; i < gridDim.x; ++i) {
            ct += __ldcg(partial + 2 * i);
            ht += __ldcg(reinterpret_cast<const unsigned long long*>(partial) + 2 * i + 1);
        }
        stats[0] = ct;
        reinterpret_cast<unsigned long long*>(stats)[1] = ht;
    }
}

int launch_batch_stats(const double* acts, size_t n, size_t B, const double* onehot, const int64_t* labels,
                       double* stats_dev, ReduceScratch& rs, cudaStream_t stream) {
    const unsigned grid = B ? cdiv(B, 256) : 1;
    RCN_TRY(rs.ensure(((size_t)2 * grid + 2048) * sizeof(double), stream));
    // shares the partial region with bias_grad_kernel (stream-ordered, each consumes its partials before it ends);
    // ticket 1023 is reserved for this kernel
    RCN_LAUNCH("batch_stats_kernel", stream,
               batch_stats_kernel<<<grid, 256, 0, stream>>>(acts, (int)n, B, onehot, labels, stats_dev, rs.partials(), rs.tickets() + 1023));
    return RCN_OK;
}

// Softmax cross-entropy head (launch_softmax_xent_head): one warp per sample (grid-stride), softmax_xent_warp's arithmetic,
// in place over the logits.  Hits and labels are decided on z, not on p: exp rounding can make distinct logits equal
// probabilities (z = (0, 2^-60) gives p = (0.5, 0.5)).  The argmax follows argmax_last_kernel's sequential rule exactly,
// NaN included: after the last NaN q the scan restarts at q + 1 (the label is q itself when q = n - 1).  Each warp adds its
// samples' costs in order, warp 0..7 sums are added in order per CTA, and the last CTA to arrive adds the per-CTA partials in
// CTA order (batch_stats_kernel's scheme: deterministic for a given B) and resets the ticket for the next launch.
__global__ void __launch_bounds__(256) softmax_xent_head_kernel(double* __restrict__ z, int n, size_t B,
                                                               const int64_t* __restrict__ labels, double* __restrict__ delta,
                                                               int64_t* __restrict__ labels_out, double* __restrict__ stats,
                                                               double* __restrict__ partial, unsigned* __restrict__ ticket) {
    __shared__ double sc[8];
    __shared__ unsigned long long sh[8];
    __shared__ bool s_last;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const size_t warp = (blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5;
    const size_t n_warps = ((size_t)gridDim.x * blockDim.x) >> 5;
    double cost = 0.0;
    unsigned long long hits = 0;
    for (size_t b = warp; b < B; b += n_warps) {
        double* zb = z + b * n;
        const int64_t lab = labels ? labels[b] : -1;
        int q = -1;                                       // last NaN logit
        int best = -1;
        if (labels_out) {
            for (int i = lane; i < n; i += 32) if (zb[i] != zb[i]) q = i;
            q = __reduce_max_sync(0xffffffffu, q);
            if (q >= 0 && q + 1 < n) {                    // last-max-wins over (q, n), which holds no NaN
                double mx = -INFINITY;
                for (int i = q + 1 + lane; i < n; i += 32) mx = fmax(mx, zb[i]);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
                for (int i = q + 1 + lane; i < n; i += 32) if (zb[i] == mx) best = i;
            } else if (q >= 0) {
                best = q;
            }
        }
        bool ok = true;
        int at_max = -1;
        const auto target = [&](int i) { return lab == (int64_t)i ? 1.0 : 0.0; };
        const auto visit = [&](int i, double zi, double m, double p, double d) {
            zb[i] = p;
            if (delta) delta[b * n + i] = d;
            ok = ok && ((zi == m) == (lab == (int64_t)i));   // {i : z_i = max z} == {label}
            if (zi == m) at_max = i;
        };
        const double l = softmax_xent_warp(zb, n, lane, target, visit);
        if (labels_out) {
            if (q < 0) best = at_max;
            best = __reduce_max_sync(0xffffffffu, best);
            if (lane == 0) labels_out[b] = best;
        }
        const bool hit = __all_sync(0xffffffffu, ok);
        cost += l;
        hits += hit ? 1ull : 0ull;
    }
    if (!stats) return;
    if (lane == 0) { sc[w] = cost; sh[w] = hits; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double ct = 0.0;
        unsigned long long ht = 0;
        for (int i = 0; i < 8; ++i) { ct += sc[i]; ht += sh[i]; }
        partial[2 * blockIdx.x] = ct;
        reinterpret_cast<unsigned long long*>(partial)[2 * blockIdx.x + 1] = ht;
        __threadfence();
        const unsigned t = atomicAdd(ticket, 1u);
        s_last = (t == gridDim.x - 1);
        if (s_last) *ticket = 0;
    }
    __syncthreads();
    if (s_last && threadIdx.x == 0) {
        __threadfence();
        double ct = 0.0;
        unsigned long long ht = 0;
        for (unsigned i = 0; i < gridDim.x; ++i) {
            ct += __ldcg(partial + 2 * i);
            ht += __ldcg(reinterpret_cast<const unsigned long long*>(partial) + 2 * i + 1);
        }
        stats[0] = ct;
        reinterpret_cast<unsigned long long*>(stats)[1] = ht;
    }
}

int launch_softmax_xent_head(double* z, size_t n, size_t B, const int64_t* labels, double* delta, int64_t* labels_out,
                             double* stats_dev, ReduceScratch& rs, cudaStream_t stream) {
    if (n == 0 || n > 0x7fffffff) return fail(RCN_ERR_INVALID, "softmax head over %zu classes", n);
    if (stats_dev && !labels) return fail(RCN_ERR_INVALID, "internal: head statistics need labels");
    if (B == 0) return RCN_OK;
    unsigned grid = cdiv(B, 8);
    if (grid > kNumSMs * 8) grid = kNumSMs * 8;
    // the partial region and ticket 1023 of batch_stats_kernel, which this kernel replaces on the softmax head
    RCN_TRY(rs.ensure(((size_t)2 * grid + 2048) * sizeof(double), stream));
    RCN_LAUNCH("softmax_xent_head_kernel", stream,
               softmax_xent_head_kernel<<<grid, 256, 0, stream>>>(z, (int)n, B, labels, delta, labels_out, stats_dev, rs.partials(),
                                                                  rs.tickets() + 1023));
    return RCN_OK;
}

}  // namespace rcn

using namespace rcn;

extern "C" int rcn_cuda_ext_gemm_f64(int device, void* cuda_stream, const double* A, size_t lda, int a_kcontig, const double* B,
                                     size_t ldb, int b_kcontig, size_t M, size_t N, size_t K, int impl, double* C) {
    if (!A || !B || !C) return fail(RCN_ERR_INVALID, "null pointer");
    if (M == 0 || N == 0) return RCN_OK;
    if (M > 0x7fffffff || N > 0x7fffffff || K > 0x7fffffff) return fail(RCN_ERR_INVALID, "GEMM dimension too large");
    if (impl != 0 && impl != 1) return fail(RCN_ERR_INVALID, "impl must be 0 (DMMA) or 1 (tcgen05 integer slices)");
    OpCtx c;
    RCN_TRY(c.enter(device, cuda_stream));
    const size_t a_elems = a_kcontig ? (M - 1) * lda + K : (K ? (K - 1) * lda + M : 0);
    const size_t b_elems = b_kcontig ? (N - 1) * ldb + K : (K ? (K - 1) * ldb + N : 0);
    const void *a_dev = nullptr, *b_dev = nullptr; void* c_dev = nullptr; bool host = false;
    RCN_TRY(c.in(A, a_elems * 8, tl_op_in, &a_dev));
    RCN_TRY(c.in(B, b_elems * 8, tl_op_in2, &b_dev));
    RCN_TRY(c.out(C, M * N * 8, tl_op_out, &c_dev, &host));
    EpiStore epi{(double*)c_dev, (int)M, 0};
    if (impl == 1) {
        if (!ozaki_available()) return fail(RCN_ERR_CUDA, "tensor-map encoding is not available from this driver");
        static thread_local OzakiWorkspace ws;
        const OzOperand oa{(const double*)a_dev, lda, a_kcontig != 0}, ob{(const double*)b_dev, ldb, b_kcontig != 0};
        RCN_TRY(launch_gemm_ozaki("ext_gemm_f64(tcgen05 int8 slices)", oa, ob, (int)M, (int)N, (int)K, epi, ws, c.stream));
    } else {
        int splits = 1, kps;
        split_plan((int)K, splits, kps);
#define RCN_EXT_GEMM(AKC, BKC)                                                                       \
        {                                                                                            \
            const DenseLoader<AKC> la{(const double*)a_dev, (int)lda, (int)M};                       \
            const DenseLoader<BKC> lb{(const double*)b_dev, (int)ldb, (int)N};                       \
            RCN_TRY(launch_gemm_tiles("ext_gemm_f64(dmma)", la, lb, (int)M, (int)N, (int)K, 1, kps, epi, c.stream)); \
        }
        if (a_kcontig && b_kcontig) RCN_EXT_GEMM(true, true)
        else if (a_kcontig) RCN_EXT_GEMM(true, false)
        else if (b_kcontig) RCN_EXT_GEMM(false, true)
        else RCN_EXT_GEMM(false, false)
#undef RCN_EXT_GEMM
    }
    return c.finish(C, c_dev, M * N * 8, host);
}


