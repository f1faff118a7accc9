// conv.cu -- EXTENSION (not in the reference): learned multi-channel convolution forward / backward-data /
// backward-weight in f64, NHWC.
//
// rcn's own "convolution" is four fixed Sobel operators per map (rcn/src/utils/kernel.rs:38-53, rcn/src/rcn.rs:
// 319-341) with no weights and no backward pass; BASELINE.json's north_star additionally names learned convolution
// layers (SURVEY.md section 8a row x1).  Conventions extend the reference's: cross-correlation without kernel flip
// and Padding::{None, Same} as in Convolve2D::convolve_2d (kernel.rs:110-194, with the un-quirked zero padding of
// kh/2, kw/2 pinned by kernel.rs:434-441).  Checked against oracle/ext_oracle.cpp ("parity unpinned").
//
// Layout: x[b][y][x][ci], w[co][ky][kx][ci], y[b][oy][ox][co], all f64.
//
//   forward          Y(co, pix)  = sum_k W(co, k) * im2col(X)(k, pix)          k = (ky, kx, ci)
//   backward-data    dX(ci, pix) = sum_k W'(ci, k) * im2col(dZ)(k, pix)        k = (ky', kx', co), W' = flipped/transposed W
//   backward-weight  dW(co, k)   = sum_pix dZ(co, pix) * im2col(X)(pix, k)     split over pixels, fixed-order combine
//
// All three are implicit GEMMs on the f64 tensor path (DMMA, gemm_f64.cuh): the im2col operand is gathered tile by
// tile by a loader policy (cp.async with zero fill for the padding), never materialised.  Small-channel first
// layers (Ci*kh*kw <= 64, e.g. 1- or 3-channel images) are not dense contractions: they run a direct kernel that
// stages the input halo tile and the weights in shared memory (north_star: "small-channel first layers ... run as
// coalesced, vectorised, shared-memory-staged kernels").
#include "conv.cuh"
#include "dense.cuh"
#include "gemm_f64.cuh"
#include "opctx.cuh"
#include "ozaki.cuh"

namespace rcn {

__device__ __forceinline__ double act_forward(double z, int act) {
    if (act == ACT_RELU) return z >= 0.0 ? z : 0.0;              // kernel.rs:209-216 rule
    if (act == ACT_SIGMOID) return 1.0 / (1.0 + exp(-z));        // rcn.rs:478-483
    return z;
}
__device__ __forceinline__ double act_backward_from_output(double y, int act) {
    if (act == ACT_RELU) return y > 0.0 ? 1.0 : 0.0;
    if (act == ACT_SIGMOID) return y * (1.0 - y);                // rcn.rs:490-492
    return 1.0;
}

// B operand with rows = grid pixels and contraction k = (ky, kx, c), c fastest (forward, backward-data).
struct Im2colPixelRows {
    static constexpr bool KCONTIG = true;
    static constexpr int kPrepInts = 3;   // per row: pixel base b*Hi*Wi, oy - ph, ox - pw
    ConvGeom g;
    template <int ROWS>
    __device__ __forceinline__ void prepare(int* info, int r0, int tid) const {
        for (int r = tid; r < ROWS; r += GEMM_THREADS) {
            const int n = r0 + r;
            int base = 0, oy = -(1 << 28), ox = 0;
            if (n < g.n_pix) {
                const int b = n / (g.Ho * g.Wo);
                const int rem = n - b * g.Ho * g.Wo;
                oy = rem / g.Wo;
                ox = rem - oy * g.Wo;
                base = b * g.Hi * g.Wi;
                oy -= g.ph; ox -= g.pw;
            }
            info[3 * r] = base; info[3 * r + 1] = oy; info[3 * r + 2] = ox;
        }
    }
    template <int ROWS>
    __device__ __forceinline__ void load_tile(double* s, const int* info, int, int k0, int kmax, int tid) const {
        using TL = TileLayout<ROWS, true>;
        static_assert(GEMM_THREADS % KT == 0, "kk must be fixed per thread");
        const int kk = tid % KT;
        const int k = k0 + kk;
        const bool kok = k < kmax;
        const int tap = k / g.C, c = k - tap * g.C;
        const int ky = tap / g.kw, kx = tap - ky * g.kw;
#pragma unroll
        for (int i = 0; i < ROWS * KT / GEMM_THREADS; ++i) {
            const int r = tid / KT + i * (GEMM_THREADS / KT);
            const int iy = info[3 * r + 1] + ky, ix = info[3 * r + 2] + kx;
            const bool ok = kok && (unsigned)iy < (unsigned)g.Hi && (unsigned)ix < (unsigned)g.Wi;
            const size_t off = ((size_t)(info[3 * r] + iy * g.Wi + ix)) * g.C + c;
            cp_async8(s + TL::idx(r, kk), ok ? g.t + off : g.t, ok ? 8 : 0);
        }
    }
};

// B operand with rows = weight-gradient columns (ky, kx, c) and contraction over grid pixels (backward-weight).
struct Im2colPixelK {
    static constexpr bool KCONTIG = false;
    static constexpr int kPrepInts = 3;   // per row: ky - ph, kx - pw, c  (c < 0: column out of range)
    ConvGeom g;
    template <int ROWS>
    __device__ __forceinline__ void prepare(int* info, int r0, int tid) const {
        for (int r = tid; r < ROWS; r += GEMM_THREADS) {
            const int col = r0 + r;
            int dy = 0, dx = 0, c = -1;
            if (col < g.n_k) {
                const int tap = col / g.C;
                c = col - tap * g.C;
                const int ky = tap / g.kw;
                dy = ky - g.ph; dx = (tap - ky * g.kw) - g.pw;
            }
            info[3 * r] = dy; info[3 * r + 1] = dx; info[3 * r + 2] = c;
        }
    }
    template <int ROWS>
    __device__ __forceinline__ void load_tile(double* s, const int* info, int, int k0, int kmax, int tid) const {
        using TL = TileLayout<ROWS, false>;
        static_assert(GEMM_THREADS % ROWS == 0, "the row must be fixed per thread");
        const int r = tid % ROWS;
        const int dy = info[3 * r], dx = info[3 * r + 1], c = info[3 * r + 2];
#pragma unroll
        for (int i = 0; i < ROWS * KT / GEMM_THREADS; ++i) {
            const int kk = tid / ROWS + i * (GEMM_THREADS / ROWS);
            const int pix = k0 + kk;
            const int b = pix / (g.Ho * g.Wo);
            const int rem = pix - b * g.Ho * g.Wo;
            const int oy = rem / g.Wo, ox = rem - oy * g.Wo;
            const int iy = oy + dy, ix = ox + dx;
            const bool ok = c >= 0 && pix < kmax && (unsigned)iy < (unsigned)g.Hi && (unsigned)ix < (unsigned)g.Wi;
            const size_t off = ((size_t)((b * g.Hi + iy) * g.Wi + ix)) * g.C + c;
            cp_async8(s + TL::idx(r, kk), ok ? g.t + off : g.t, ok ? 8 : 0);
        }
    }
};

// ---- epilogues ---------------------------------------------------------------------------------------------------
struct EpiConvForward {   // y[pix*Co + co] = act(acc + bias[co])
    const double* bias; double* y; int Co, act;
    __device__ __forceinline__ void operator()(int m, int n, double v) const {
        if (bias) v += bias[m];
        y[(size_t)n * Co + m] = act_forward(v, act);
    }
};
struct EpiConvBackData {  // dx[pix*Ci + ci] = acc * act'(y_prev)
    const double* y_prev; double* dx; int Ci, act;
    __device__ __forceinline__ void operator()(int m, int n, double v) const {
        const size_t o = (size_t)n * Ci + m;
        if (y_prev) v *= act_backward_from_output(y_prev[o], act);
        dx[o] = v;
    }
};
struct EpiConvWeight {    // split-K partial (or final) of dW in [co][k] order
    double* out; int K; size_t split_stride;
    __device__ __forceinline__ void operator()(int m, int n, double v) const {
        out[(size_t)blockIdx.z * split_stride + (size_t)m * K + n] = v;
    }
};

// tcgen05 path (ozaki.cuh): grid pixels are the 128-row M side, channels the N side
struct EpiConvForwardT {   // y[pix*Co + co] = act(acc + bias[co])
    const double* bias; double* y; int Co, act;
    __device__ __forceinline__ void operator()(int m, int n, double v) const {
        if (bias) v += __ldg(bias + n);
        y[(size_t)m * Co + n] = act_forward(v, act);
    }
};
struct EpiConvBackDataT {  // dx[pix*Ci + ci] = acc * act'(y_prev)
    const double* y_prev; double* dx; int Ci, act;
    __device__ __forceinline__ void operator()(int m, int n, double v) const {
        const size_t o = (size_t)m * Ci + n;
        if (y_prev) v *= act_backward_from_output(y_prev[o], act);
        dx[o] = v;
    }
};

// w'[ci][ky'][kx'][co] = w[co][kh-1-ky'][kw-1-kx'][ci]
__global__ void conv_flip_weights_kernel(const double* __restrict__ w, int Co, int kh, int kw, int Ci, double* __restrict__ wt) {
    const int n = Co * kh * kw * Ci;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int co = i % Co;
        int r = i / Co;
        const int kx = r % kw; r /= kw;
        const int ky = r % kh;
        const int ci = r / kh;
        wt[i] = w[(((size_t)co * kh + (kh - 1 - ky)) * kw + (kw - 1 - kx)) * Ci + ci];
    }
}

__global__ void activation_backward_kernel(const double* __restrict__ y, const double* __restrict__ dy, size_t n, int act,
                                           double* __restrict__ dz) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        dz[i] = dy[i] * act_backward_from_output(y[i], act);
}

// ---- direct kernel for small-channel first layers --------------------------------------------------------------------
// One CTA = a 16 x 16 tile of output pixels of one image, all output channels.  The input halo tile
// ((16+kh-1) x (16+kw-1) x Ci) and the whole weight tensor are staged in shared memory (coalesced row runs); each
// thread owns one pixel and produces the output channels eight at a time (weights are warp-uniform broadcasts).
// The pixel type is a template parameter: u8 images (one channel) are read as they are stored.
constexpr int DT = 16;
template <typename Px>
__device__ __forceinline__ void conv2d_direct_small(const Px* __restrict__ x, int H, int W, int Ci, const double* __restrict__ w,
                                                    const double* __restrict__ bias, int Co, int kh, int kw, int ph, int pw, int Ho,
                                                    int Wo, int act, double* __restrict__ y) {
    extern __shared__ __align__(16) double sm_direct[];
    const int th = DT + kh - 1, tw = DT + kw - 1;
    const int kk = kh * kw * Ci;
    double* sx = sm_direct;                 // [th][tw][Ci]
    double* sw = sm_direct + th * tw * Ci;  // [Co][kh][kw][Ci]
    const int tid = threadIdx.x;
    const int b = blockIdx.z;
    const int oy0 = blockIdx.y * DT, ox0 = blockIdx.x * DT;
    for (int i = tid; i < Co * kk; i += DT * DT) sw[i] = __ldg(w + i);
    const int row_len = tw * Ci;
    for (int i = tid; i < th * row_len; i += DT * DT) {
        const int ry = i / row_len, rx = i - ry * row_len;
        const int iy = oy0 + ry - ph;
        const int ix = ox0 - pw + rx / Ci;
        const bool ok = (unsigned)iy < (unsigned)H && (unsigned)ix < (unsigned)W;
        sx[i] = ok ? (double)__ldg(x + (((long long)b * H + iy) * W + (ox0 - pw)) * Ci + rx) : 0.0;
    }
    __syncthreads();
    const int ty = tid / DT, tx = tid % DT;
    const int oy = oy0 + ty, ox = ox0 + tx;
    if (oy >= Ho || ox >= Wo) return;
    double* yo = y + (((size_t)b * Ho + oy) * Wo + ox) * Co;
    for (int co0 = 0; co0 < Co; co0 += 8) {
        double acc[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] = 0.0;
        for (int ky = 0; ky < kh; ++ky)
            for (int q = 0; q < kw * Ci; ++q) {       // (kx, ci) run is contiguous in both the tile row and the weights
                const double xv = sx[((ty + ky) * tw + tx) * Ci + q];
                const double* wp = sw + (size_t)co0 * kk + ky * kw * Ci + q;
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    if (co0 + j < Co) acc[j] = fma(xv, wp[j * kk], acc[j]);
            }
#pragma unroll
        for (int j = 0; j < 8; ++j)
            if (co0 + j < Co) {
                double v = acc[j];
                if (bias) v += __ldg(bias + co0 + j);
                yo[co0 + j] = act_forward(v, act);
            }
    }
}
__global__ void __launch_bounds__(DT * DT) conv2d_direct_small_kernel(const double* __restrict__ x, int H, int W, int Ci,
                                                                       const double* __restrict__ w, const double* __restrict__ bias,
                                                                       int Co, int kh, int kw, int ph, int pw, int Ho, int Wo,
                                                                       int act, double* __restrict__ y) {
    conv2d_direct_small(x, H, W, Ci, w, bias, Co, kh, kw, ph, pw, Ho, Wo, act, y);
}
__global__ void __launch_bounds__(DT * DT) conv2d_direct_small_u8_kernel(const uint8_t* __restrict__ x, int H, int W, int Ci,
                                                                          const double* __restrict__ w, const double* __restrict__ bias,
                                                                          int Co, int kh, int kw, int ph, int pw, int Ho, int Wo,
                                                                          int act, double* __restrict__ y) {
    conv2d_direct_small(x, H, W, Ci, w, bias, Co, kh, kw, ph, pw, Ho, Wo, act, y);
}

// ---- host side --------------------------------------------------------------------------------------------------------
int check_conv_shape(size_t B, size_t H, size_t W, size_t Ci, size_t Co, size_t kh, size_t kw, int padding, ConvShape* s) {
    if (padding != RCN_PADDING_NONE && padding != RCN_PADDING_SAME) return fail(RCN_ERR_INVALID, "unknown padding %d", padding);
    if (Ci == 0 || Co == 0) return fail(RCN_ERR_INVALID, "zero channels");
    // same contract as Convolve2D::convolve_2d (kernel.rs:123-135)
    if (kh == 0 || kw == 0 || kh > H || kw > W)
        return fail(RCN_ERR_SHAPE, "conv2d expects 'input shape >= kernel shape > 0', received (%zu, %zu) and (%zu, %zu) respectively.", H, W, kh, kw);
    if (padding == RCN_PADDING_SAME && (kh % 2 == 0 || kw % 2 == 0))
        return fail(RCN_ERR_SHAPE, "conv2d expects kernel dimensions to be odd when padding mode set to 'SAME', got (%zu, %zu)", kh, kw);
    const bool same = padding == RCN_PADDING_SAME;
    s->B = B; s->H = H; s->W = W; s->Ci = Ci; s->Co = Co; s->kh = kh; s->kw = kw; s->padding = padding;
    s->Ho = same ? H : H - kh + 1; s->Wo = same ? W : W - kw + 1;
    s->ph = same ? (int)(kh / 2) : 0; s->pw = same ? (int)(kw / 2) : 0;
    const size_t lim = (size_t)1 << 31;
    if (B * H * W >= lim || B * s->Ho * s->Wo >= lim || kh * kw * Ci >= lim || kh * kw * Co >= lim || B * H * W * (Ci > Co ? Ci : Co) >= ((size_t)1 << 40))
        return fail(RCN_ERR_INVALID, "convolution problem too large for 32-bit pixel indices");
    return RCN_OK;
}

namespace {

// tcgen05 integer-slice implicit GEMM when the contraction is really dense (wide-channel layers: BASELINE config 4):
// >= half the SMs worth of 128-pixel x 96-channel tiles, K = kh*kw*C deep enough, enough work to amortise the gather.
bool conv_use_tc(size_t n_pix, size_t n_out, size_t K) {
    const GemmImpl impl = gemm_impl();
    if (impl == GEMM_DMMA || impl == GEMM_SIMT || !ozaki_available() || K > (size_t)OZ_MAX_K) return false;
    if (impl == GEMM_TC) return true;
    const size_t tiles = ((n_pix + OZ_BM - 1) / OZ_BM) * ((n_out + OZ_BN - 1) / OZ_BN);
    return n_out >= 32 && K >= 256 && tiles >= (size_t)kNumSMs / 2 && (double)n_pix * (double)n_out * (double)K >= 2.0e9;
}

// backward-weight contracts over the pixels (K = B*Ho*Wo, split across CTAs), so the tile count does not matter
bool conv_wgrad_use_tc(size_t Co, size_t n_k, size_t n_pix) {
    const GemmImpl impl = gemm_impl();
    if (impl == GEMM_DMMA || impl == GEMM_SIMT || !ozaki_available()) return false;
    if (impl == GEMM_TC) return true;
    return Co >= 64 && n_k >= 256 && n_pix >= 4096 && (double)Co * (double)n_k * (double)n_pix >= 2.0e9;
}

OzakiWorkspace& conv_tc_workspace() {
    static thread_local OzakiWorkspace ws[64];   // one per device this thread drives
    int dev = 0;
    cudaGetDevice(&dev);
    return ws[dev & 63];
}

bool use_direct(const ConvShape& s) {
    static const bool off = []() { const char* e = getenv("RCN_CUDA_CONV_DIRECT"); return e && e[0] == '0'; }();
    const size_t kk = s.kh * s.kw * s.Ci;
    const size_t smem = ((DT + s.kh - 1) * (DT + s.kw - 1) * s.Ci + s.Co * kk) * sizeof(double);
    return !off && kk <= 64 && smem <= 96 * 1024;
}

}  // namespace

bool conv_direct_ok(const ConvShape& s) { return use_direct(s); }

int launch_conv2d_forward_u8(const uint8_t* x, const double* w, const double* bias, const ConvShape& s, int act, double* y,
                             cudaStream_t stream) {
    if (s.B == 0) return RCN_OK;
    if (!use_direct(s) || s.Ci != 1) return fail(RCN_ERR_STATE, "internal: u8 convolution outside the direct kernel");
    if (s.B > 65535) return fail(RCN_ERR_INVALID, "batch too large for the direct convolution kernel");
    const size_t smem = ((DT + s.kh - 1) * (DT + s.kw - 1) * s.Ci + s.Co * s.kh * s.kw * s.Ci) * sizeof(double);
    static SmemAttrCache attr;
    if (smem > 48 * 1024 && attr.need(smem))
        RCN_CUDA_TRY(cudaFuncSetAttribute(conv2d_direct_small_u8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid(cdiv(s.Wo, DT), cdiv(s.Ho, DT), (unsigned)s.B);
    RCN_LAUNCH("conv2d_direct_small_u8_kernel", stream,
               conv2d_direct_small_u8_kernel<<<grid, DT * DT, smem, stream>>>(x, (int)s.H, (int)s.W, (int)s.Ci, w, bias, (int)s.Co,
                                                                             (int)s.kh, (int)s.kw, s.ph, s.pw, (int)s.Ho, (int)s.Wo,
                                                                             act, y));
    return RCN_OK;
}

int launch_activation_backward(const double* y, const double* dy, size_t n, int act, double* dz, cudaStream_t stream) {
    if (n == 0) return RCN_OK;
    unsigned grid = cdiv(n, 256);
    if (grid > kNumSMs * 8) grid = kNumSMs * 8;
    RCN_LAUNCH("activation_backward_kernel", stream,
               activation_backward_kernel<<<grid, 256, 0, stream>>>(y, dy, n, act, dz));
    return RCN_OK;
}

int launch_conv2d_forward(const double* x, const double* w, const double* bias, const ConvShape& s, int act, double* y,
                          cudaStream_t stream, OzakiWorkspace* tw) {
    if (s.B == 0) return RCN_OK;
    if (use_direct(s)) {
        const size_t kk = s.kh * s.kw * s.Ci;
        const size_t smem = ((DT + s.kh - 1) * (DT + s.kw - 1) * s.Ci + s.Co * kk) * sizeof(double);
        static SmemAttrCache attr;
        if (smem > 48 * 1024 && attr.need(smem))
            RCN_CUDA_TRY(cudaFuncSetAttribute(conv2d_direct_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        if (s.B > 65535) return fail(RCN_ERR_INVALID, "batch too large for the direct convolution kernel");
        dim3 grid(cdiv(s.Wo, DT), cdiv(s.Ho, DT), (unsigned)s.B);
        RCN_LAUNCH("conv2d_direct_small_kernel", stream,
                   conv2d_direct_small_kernel<<<grid, DT * DT, smem, stream>>>(x, (int)s.H, (int)s.W, (int)s.Ci, w, bias, (int)s.Co,
                                                                                (int)s.kh, (int)s.kw, s.ph, s.pw, (int)s.Ho,
                                                                                (int)s.Wo, act, y));
        return RCN_OK;
    }
    const int M = (int)s.Co, N = (int)(s.B * s.Ho * s.Wo), K = (int)(s.kh * s.kw * s.Ci);
    const ConvGeom geom{x, (int)s.H, (int)s.W, (int)s.Ci, (int)s.Ho, (int)s.Wo, (int)s.kh, (int)s.kw, s.ph, s.pw, N, K};
    if (conv_use_tc((size_t)N, (size_t)M, (size_t)K)) {
        OzakiWorkspace& ows = tw ? *tw : conv_tc_workspace();
        const EpiConvForwardT epi{bias, y, M, act};
        if (ozaki_conv_tma_ok(geom))   // im2col by TMA: the tensor is sliced once, taps are shifted boxes
            return launch_conv_ozaki("conv2d_forward_igemm(tcgen05 int8 slices, TMA im2col)", geom, (int)s.B, w, M, epi,
                                     ows, stream);
        OzOperand oa{x, 0, true};                 // im2col rows gathered straight into int8 digit planes
        oa.gather = 1; oa.g = geom;
        const OzOperand ob{w, (size_t)K, true};   // w[co][k]
        return launch_gemm_ozaki("conv2d_forward_igemm(tcgen05 int8 slices)", oa, ob, N, M, K, epi, ows, stream);
    }
    const DenseLoader<true> la{w, K, M};
    const Im2colPixelRows lb{geom};
    const EpiConvForward epi{bias, y, M, act};
    int splits = 1, kps;
    split_plan(K, splits, kps);
    return launch_gemm_tiles("conv2d_forward_igemm", la, lb, M, N, K, 1, kps, epi, stream);
}

int launch_conv2d_backward_data(const double* dz, const double* w, const ConvShape& s, const double* y_prev, int act_prev,
                                double* dx, DevBuf& ws, cudaStream_t stream, OzakiWorkspace* tw) {
    if (s.B == 0) return RCN_OK;
    const size_t nw = s.Co * s.kh * s.kw * s.Ci;
    RCN_TRY(ws.reserve(nw * sizeof(double)));
    unsigned grid = cdiv(nw, 256);
    if (grid > kNumSMs * 4) grid = kNumSMs * 4;
    RCN_LAUNCH("conv_flip_weights_kernel", stream,
               conv_flip_weights_kernel<<<grid, 256, 0, stream>>>(w, (int)s.Co, (int)s.kh, (int)s.kw, (int)s.Ci, ws.as<double>()));
    const int M = (int)s.Ci, N = (int)(s.B * s.H * s.W), K = (int)(s.kh * s.kw * s.Co);
    // gather from dz [B][Ho][Wo][Co] over the INPUT pixel grid with the complementary padding
    const ConvGeom geom{dz, (int)s.Ho, (int)s.Wo, (int)s.Co, (int)s.H, (int)s.W, (int)s.kh, (int)s.kw,
                        (int)s.kh - 1 - s.ph, (int)s.kw - 1 - s.pw, N, K};
    if (conv_use_tc((size_t)N, (size_t)M, (size_t)K)) {
        OzakiWorkspace& ows = tw ? *tw : conv_tc_workspace();
        const EpiConvBackDataT epi{y_prev, dx, M, act_prev};
        if (ozaki_conv_tma_ok(geom))
            return launch_conv_ozaki("conv2d_backward_data_igemm(tcgen05 int8 slices, TMA im2col)", geom, (int)s.B, ws.as<double>(), M,
                                     epi, ows, stream);
        OzOperand oa{dz, 0, true};
        oa.gather = 1; oa.g = geom;
        const OzOperand ob{ws.as<double>(), (size_t)K, true};   // w'[ci][k]
        return launch_gemm_ozaki("conv2d_backward_data_igemm(tcgen05 int8 slices)", oa, ob, N, M, K, epi, ows, stream);
    }
    const DenseLoader<true> la{ws.as<double>(), K, M};
    const Im2colPixelRows lb{geom};
    const EpiConvBackData epi{y_prev, dx, M, act_prev};
    int splits = 1, kps;
    split_plan(K, splits, kps);
    return launch_gemm_tiles("conv2d_backward_data_igemm", la, lb, M, N, K, 1, kps, epi, stream);
}

int launch_conv2d_backward_weight(const double* x, const double* dz, const ConvShape& s, double* dw, double* db, DevBuf& ws,
                                  cudaStream_t stream, OzakiWorkspace* tw_in, ReduceScratch* rs) {
    const int M = (int)s.Co, N = (int)(s.kh * s.kw * s.Ci), Kc = (int)(s.B * s.Ho * s.Wo);
    if (Kc == 0) {
        RCN_CUDA_TRY(cudaMemsetAsync(dw, 0, (size_t)M * N * sizeof(double), stream));
        if (db) RCN_CUDA_TRY(cudaMemsetAsync(db, 0, (size_t)M * sizeof(double), stream));
        return RCN_OK;
    }
    if (conv_wgrad_use_tc((size_t)M, (size_t)N, (size_t)Kc)) {
        // contraction over the grid pixels: dz columns (co) x im2col columns (ky, kx, ci), both gathered straight into
        // digit planes with per-row scales over ALL pixels; split-K keeps each CTA's contraction inside the exact int32
        // range and fills the machine; partials are combined in split order (deterministic)
        OzakiWorkspace& tw = tw_in ? *tw_in : conv_tc_workspace();
        const int splits = ozaki_plan_splits(M, N, Kc);
        OzOperand oa{dz, (size_t)M, false};                      // element (co, pix) at dz[pix*Co + co]
        OzOperand ob{x, 0, false};
        ob.gather = 2;
        ob.g = ConvGeom{x, (int)s.H, (int)s.W, (int)s.Ci, (int)s.Ho, (int)s.Wo, (int)s.kh, (int)s.kw, s.ph, s.pw, Kc, N};
        if (splits == 1) {
            const EpiOzSplitStore epi{dw, (size_t)N, 1, 0};
            RCN_TRY(launch_gemm_ozaki("conv2d_backward_weight_igemm(tcgen05 int8 slices)", oa, ob, M, N, Kc, epi, tw, stream, 1));
        } else {
            RCN_TRY(tw.partials.reserve((size_t)splits * M * N * sizeof(double)));
            const EpiOzSplitStore epi{tw.partials.as<double>(), (size_t)N, 1, (size_t)M * N};
            RCN_TRY(launch_gemm_ozaki("conv2d_backward_weight_igemm(tcgen05 int8 slices)", oa, ob, M, N, Kc, epi, tw, stream, splits));
            RCN_TRY(launch_reduce_splits(tw.partials.as<double>(), splits, (size_t)M * N, dw, stream));
        }
        if (db && rs) RCN_TRY(launch_bias_grad(dz, (size_t)M, (size_t)Kc, db, *rs, stream));
        else if (db) {
            static thread_local ReduceScratch tl_rs2[64];
            int dev = 0;
            RCN_CUDA_TRY(cudaGetDevice(&dev));
            RCN_TRY(launch_bias_grad(dz, (size_t)M, (size_t)Kc, db, tl_rs2[dev & 63], stream));
        }
        return RCN_OK;
    }
    size_t tiles;
    if (M <= 32) tiles = (size_t)cdiv(M, 32) * cdiv(N, 128);
    else {
        tiles = (size_t)cdiv(M, 128) * cdiv(N, 128);
        if (tiles < (size_t)kNumSMs) tiles = (size_t)cdiv(M, 64) * cdiv(N, 64);
    }
    int splits = 1;
    if (tiles < (size_t)kNumSMs) {
        splits = (int)((2 * kNumSMs + tiles - 1) / tiles);
        const int max_splits = Kc / 64 > 0 ? Kc / 64 : 1;
        if (splits > max_splits) splits = max_splits;
        if (splits > 128) splits = 128;
    }
    int kps;
    split_plan(Kc, splits, kps);
    // big tiles are chosen by tile count INCLUDING splits; recompute as launch_gemm_tiles will see it
    const DenseLoader<false> la{dz, M, M};
    const Im2colPixelK lb{ConvGeom{x, (int)s.H, (int)s.W, (int)s.Ci, (int)s.Ho, (int)s.Wo, (int)s.kh, (int)s.kw, s.ph, s.pw, Kc, N}};
    if (splits == 1) {
        const EpiConvWeight epi{dw, N, 0};
        RCN_TRY(launch_gemm_tiles("conv2d_backward_weight_igemm", la, lb, M, N, Kc, 1, kps, epi, stream));
    } else {
        RCN_TRY(ws.reserve((size_t)splits * M * N * sizeof(double)));
        const EpiConvWeight epi{ws.as<double>(), N, (size_t)M * N};
        RCN_TRY(launch_gemm_tiles("conv2d_backward_weight_igemm", la, lb, M, N, Kc, splits, kps, epi, stream));
        RCN_TRY(launch_reduce_splits(ws.as<double>(), splits, (size_t)M * N, dw, stream));
    }
    if (db && rs) RCN_TRY(launch_bias_grad(dz, (size_t)M, (size_t)Kc, db, *rs, stream));
    else if (db) {
        static thread_local ReduceScratch tl_rs[64];   // one per device this thread drives
        int dev = 0;
        RCN_CUDA_TRY(cudaGetDevice(&dev));
        RCN_TRY(launch_bias_grad(dz, (size_t)M, (size_t)Kc, db, tl_rs[dev & 63], stream));
    }
    return RCN_OK;
}

}  // namespace rcn

using namespace rcn;

extern "C" {

int rcn_cuda_ext_conv2d_forward(int device, void* cuda_stream, const double* x, size_t B, size_t H, size_t W, size_t Ci,
                                const double* w, const double* bias, size_t Co, size_t kh, size_t kw, int padding,
                                int activation, double* y) {
    if (!x || !w || !y) return fail(RCN_ERR_INVALID, "null pointer");
    if (activation < ACT_NONE || activation > ACT_SIGMOID) return fail(RCN_ERR_INVALID, "unknown activation %d", activation);
    ConvShape s;
    RCN_TRY(check_conv_shape(B, H, W, Ci, Co, kh, kw, padding, &s));
    OpCtx c;
    RCN_TRY(c.enter(device, cuda_stream));
    const void *x_dev = nullptr, *w_dev = nullptr, *b_dev = nullptr; void* y_dev = nullptr; bool host = false;
    const size_t ny = B * s.Ho * s.Wo * Co;
    RCN_TRY(c.in(x, B * H * W * Ci * 8, tl_op_in, &x_dev));
    RCN_TRY(c.in(w, Co * kh * kw * Ci * 8, tl_op_k, &w_dev));
    if (bias) RCN_TRY(c.in(bias, Co * 8, tl_op_aux, &b_dev));
    RCN_TRY(c.out(y, ny * 8, tl_op_out, &y_dev, &host));
    RCN_TRY(launch_conv2d_forward((const double*)x_dev, (const double*)w_dev, (const double*)b_dev, s, activation, (double*)y_dev, c.stream));
    return c.finish(y, y_dev, ny * 8, host);
}

int rcn_cuda_ext_activation_backward(int device, void* cuda_stream, const double* y, const double* dy, size_t n,
                                     int activation, double* dz) {
    if (n == 0) return RCN_OK;
    if (!y || !dy || !dz) return fail(RCN_ERR_INVALID, "null pointer");
    if (activation < ACT_NONE || activation > ACT_SIGMOID) return fail(RCN_ERR_INVALID, "unknown activation %d", activation);
    OpCtx c;
    RCN_TRY(c.enter(device, cuda_stream));
    const void *y_dev = nullptr, *dy_dev = nullptr; void* o_dev = nullptr; bool host = false;
    RCN_TRY(c.in(y, n * 8, tl_op_in, &y_dev));
    RCN_TRY(c.in(dy, n * 8, tl_op_in2, &dy_dev));
    RCN_TRY(c.out(dz, n * 8, tl_op_out, &o_dev, &host));
    RCN_TRY(launch_activation_backward((const double*)y_dev, (const double*)dy_dev, n, activation, (double*)o_dev, c.stream));
    return c.finish(dz, o_dev, n * 8, host);
}

int rcn_cuda_ext_conv2d_backward_data(int device, void* cuda_stream, const double* dz, size_t B, size_t H, size_t W,
                                      size_t Ci, const double* w, size_t Co, size_t kh, size_t kw, int padding,
                                      const double* y_prev, int activation_prev, double* dx) {
    if (!dz || !w || !dx) return fail(RCN_ERR_INVALID, "null pointer");
    if (activation_prev < ACT_NONE || activation_prev > ACT_SIGMOID) return fail(RCN_ERR_INVALID, "unknown activation %d", activation_prev);
    ConvShape s;
    RCN_TRY(check_conv_shape(B, H, W, Ci, Co, kh, kw, padding, &s));
    OpCtx c;
    RCN_TRY(c.enter(device, cuda_stream));
    const void *dz_dev = nullptr, *w_dev = nullptr, *yp_dev = nullptr; void* dx_dev = nullptr; bool host = false;
    const size_t nx = B * H * W * Ci;
    RCN_TRY(c.in(dz, B * s.Ho * s.Wo * Co * 8, tl_op_in, &dz_dev));
    RCN_TRY(c.in(w, Co * kh * kw * Ci * 8, tl_op_k, &w_dev));
    if (y_prev) RCN_TRY(c.in(y_prev, nx * 8, tl_op_in2, &yp_dev));
    RCN_TRY(c.out(dx, nx * 8, tl_op_out, &dx_dev, &host));
    RCN_TRY(launch_conv2d_backward_data((const double*)dz_dev, (const double*)w_dev, s, (const double*)yp_dev, activation_prev,
                                        (double*)dx_dev, tl_op_ws, c.stream));
    return c.finish(dx, dx_dev, nx * 8, host);
}

int rcn_cuda_ext_conv2d_backward_weight(int device, void* cuda_stream, const double* x, const double* dz, size_t B, size_t H,
                                        size_t W, size_t Ci, size_t Co, size_t kh, size_t kw, int padding, double* dw,
                                        double* db) {
    if (!x || !dz || !dw) return fail(RCN_ERR_INVALID, "null pointer");
    ConvShape s;
    RCN_TRY(check_conv_shape(B, H, W, Ci, Co, kh, kw, padding, &s));
    OpCtx c;
    RCN_TRY(c.enter(device, cuda_stream));
    const void *x_dev = nullptr, *dz_dev = nullptr; void *dw_dev = nullptr, *db_dev = nullptr; bool host_w = false, host_b = false;
    const size_t nw = Co * kh * kw * Ci;
    RCN_TRY(c.in(x, B * H * W * Ci * 8, tl_op_in, &x_dev));
    RCN_TRY(c.in(dz, B * s.Ho * s.Wo * Co * 8, tl_op_in2, &dz_dev));
    RCN_TRY(c.out(dw, nw * 8, tl_op_out, &dw_dev, &host_w));
    if (db) RCN_TRY(c.out(db, Co * 8, tl_op_out2, &db_dev, &host_b));
    RCN_TRY(launch_conv2d_backward_weight((const double*)x_dev, (const double*)dz_dev, s, (double*)dw_dev, (double*)db_dev,
                                          tl_op_ws, c.stream));
    if (db && host_b) RCN_CUDA_TRY(cudaMemcpyAsync(db, db_dev, Co * 8, cudaMemcpyDeviceToHost, c.stream));
    if (host_w) return c.finish(dw, dw_dev, nw * 8, true);
    if (host_b) RCN_CUDA_TRY(cudaStreamSynchronize(c.stream));
    return RCN_OK;
}

}  // extern "C"
